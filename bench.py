#!/usr/bin/env python
"""Headline benchmark: blurry views / s (forward + backward, F sub-frames) -- BASELINE.json's metric.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2] [--impl ours|reference]

One "step" = one blurry view per GPU: sub-frame poses from the Bezier control points, all F sub-frame
renders, their mean, L1 loss against a ground-truth image, and the complete backward down to the
Gaussian parameters and the control points.  N > 1 (torchrun, one rank per GPU): every rank renders a
different blurry view over the same replicated Gaussians (views of a batch are sharded across GPUs,
weak scaling) and the Gaussian gradients are summed with one NCCL all-reduce inside the timed region.
The step is replayed as ONE CUDA graph (deblurgs_b200.graph.BlurryViewGraph; --no-graph launches it kernel by
kernel).  The same line also carries BASELINE.json's other multi-GPU shapes, measured in the same run
("other_configs"): c3 with the SUB-FRAMES of one view sharded across the ranks (strong scaling, the partial blurry
images summed by an NCCL all-reduce) and c4 with one view per rank (weak).

`--impl reference` times the reference's own implementation on the same GPU: its unmodified CUDA
extension from baseline/_ref driven by the reference's per-sub-frame Python loop (restated in
oracle/pose_torch.py because /root/reference is not present on the GPU box).
"""
import argparse
import ctypes as C
import json
import math
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from

METRIC = "blurry_views_per_s_fwd_bwd"
UNIT = "views/s"


# ------------------------------------------------------------------------------------------------
def dist_setup(n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL writes its banner / NCCL_DEBUG output to stdout by default: keep stdout for the one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
class RefCamera:
    def __init__(self, cam, device):
        self.image_width, self.image_height = cam.width, cam.height
        self.FoVx, self.FoVy, self.znear, self.zfar = cam.fovx, cam.fovy, cam.znear, cam.zfar
        self.projection_matrix = cam.projection_matrix_t().to(device)


def build_workload(config, rank, device):
    from deblurgs_b200 import synthetic
    from deblurgs_b200.motion import CameraMotionModule, GaussianParams
    P, W, H, F, order = synthetic.get_config(config)
    cam = synthetic.make_camera(W, H)
    scene = synthetic.make_scene(P, cam, seed=0).to(device)            # same Gaussians on every rank
    traj = synthetic.make_trajectory(F, order, seed=1 + rank).to(device)  # one view per rank
    gt_host = synthetic.make_target(cam, seed=2 + rank).pin_memory()
    bg = synthetic.make_background().to(device)
    gaussians = GaussianParams.from_scene(scene)
    base = torch.tensor([synthetic.BASE_SE3], dtype=torch.float32, device=device)
    cmm = CameraMotionModule([RefCamera(cam, device)], base, curve_order=order, num_subframes=F)
    with torch.no_grad():
        cmm._trans._control_points.copy_(traj.ctrl_trans[None])
        cmm._rot._control_points.copy_(traj.ctrl_rot[None])
    cmm.link_gaussian(gaussians)
    return dict(P=P, W=W, H=H, F=F, order=order, cam=cam, scene=scene, traj=traj, gt_host=gt_host, bg=bg,
                gaussians=gaussians, cmm=cmm)


def flat_grad_views(params):
    """One flat gradient buffer; every parameter's .grad is a view into it (single all-reduce)."""
    n = sum(p.numel() for p in params)
    flat = torch.zeros(n, dtype=torch.float32, device=params[0].device)
    off = 0
    for p in params:
        p.grad = flat[off:off + p.numel()].view_as(p)
        off += p.numel()
    return flat


def make_step_ours(w, world, lambda_t_smooth=0.0, use_graph=False):
    """views-dp step.  world > 1: the Gaussian gradients live in one flat buffer (deblurgs_b200.dist.FlatGradBuffer) that
    is the backward's gradient SINK: finished rows are all-reduced over NCCL (called directly, on a side stream) while
    the rest of the per-Gaussian backward still runs.  In graph mode (default) those collectives are nodes of the same
    CUDA graph as the step's kernels: one replay per step on every rank."""
    from deblurgs_b200 import dist as dd
    from deblurgs_b200.loss import blur_photometric_loss
    cmm, g = w["cmm"], w["gaussians"]
    gparams = g.parameters()
    cparams = cmm.parameters()
    sink = dd.FlatGradBuffer.for_gaussians(g) if world > 1 else None
    if sink is not None and os.environ.get("DGS_SINK_RANGES"):
        sink.n_ranges = int(os.environ["DGS_SINK_RANGES"])
    g.grad_sink = sink
    overlap = "; NCCL all-reduce of finished gradient rows on a side stream under the per-Gaussian backward" if sink is not None else ""

    if use_graph:
        from deblurgs_b200.graph import BlurryViewGraph
        graph = BlurryViewGraph(cmm, 0, w["bg"], (3, w["H"], w["W"]), lambda_t_smooth,
                                post_backward=(sink.wait if sink is not None else None),
                                caller_owned_grads=(gparams if sink is not None else ()))

        def step(gt, gt_ready=None):
            if gt_ready is not None:   # ground truth uploaded on a side stream
                torch.cuda.current_stream().wait_event(gt_ready)
            graph.gt.copy_(gt, non_blocking=True)
            return graph.replay()
        step.graph = graph
        step.mode = "cuda-graph replay (one launch per step)" + overlap.replace("; NCCL", "; inside the graph: NCCL")
        return step

    def step(gt, gt_ready=None):
        if sink is None:
            for p in gparams:
                p.grad = None
        for p in cparams:
            p.grad = None
        out = cmm.query(0, "all", background=w["bg"])
        if gt_ready is not None:   # ground truth uploaded on a side stream while the view rendered
            torch.cuda.current_stream().wait_event(gt_ready)
        # mean |blurred - gt| (+ lambda * mean |subframes[1:] - subframes[:-1]| for --loss smooth), fused
        loss = blur_photometric_loss(out["blurred"], out["subframes"], gt, lambda_t_smooth)
        loss.backward()
        if sink is not None:
            sink.wait()
        return loss
    step.graph = None
    step.mode = "kernel by kernel" + overlap
    return step


def make_step_subframe_sharded(w, world, use_graph=False):
    """One blurry view, its sub-frames sharded over the ranks (deblurgs_b200.dist.render_blurry_sharded): partial
    blurred images summed by an all-reduce, every rank evaluates the same L1 loss; the Gaussian gradients are summed
    through the gradient sink (all-reduce of finished rows under the rest of the backward), the trajectory gradients
    by one small all-reduce.  Graph mode: all of it -- collectives included -- is one CUDA-graph replay."""
    from deblurgs_b200 import dist as dd
    from deblurgs_b200.loss import blur_photometric_loss
    cmm, g = w["cmm"], w["gaussians"]
    sink = dd.FlatGradBuffer.for_gaussians(g)
    if os.environ.get("DGS_SINK_RANGES"):
        sink.n_ranges = int(os.environ["DGS_SINK_RANGES"])
    g.grad_sink = sink
    cbuf = dd.FlatGradBuffer(cmm.parameters())       # trajectory gradients: views of one flat buffer

    def finish():
        sink.wait()
        cbuf.all_reduce()

    if use_graph:
        from deblurgs_b200.graph import BlurryViewGraph

        def render(_graph):
            blurred, pkg, _ = dd.render_blurry_sharded(cmm, 0, w["bg"])
            return blurred, pkg["render"], pkg
        graph = BlurryViewGraph(cmm, 0, w["bg"], (3, w["H"], w["W"]), 0.0, pre_backward=cbuf.zero, post_backward=finish,
                                caller_owned_grads=g.parameters() + cmm.parameters(), render_fn=render)

        def step(gt, gt_ready=None):
            graph.gt.copy_(gt, non_blocking=True)
            return graph.replay()
        step.graph = graph
        step.mode = "cuda-graph replay (one launch per step; the image / gradient all-reduces are nodes of the graph)"
        return step

    def step(gt, gt_ready=None):
        cbuf.zero()
        blurred, pkg, _ = dd.render_blurry_sharded(cmm, 0, w["bg"])
        loss = blur_photometric_loss(blurred, pkg["render"], gt, 0.0)
        loss.backward()
        finish()
        return loss
    step.graph = None
    step.mode = "kernel by kernel"
    return step


def make_step_reference(w, lambda_t_smooth=0.0):
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    from oracle import pose_torch as pt   # the reference's Python loop, restated (test infrastructure)
    cmm, g, cam = w["cmm"], w["gaussians"], w["cam"]
    ref_cam = cmm.original_cam[0]
    params = g.parameters() + cmm.parameters()

    def render(view, proj, center, bg):   # gaussian_renderer/__init__.py:18-90
        xyz = g.get_xyz
        screenspace_points = torch.zeros_like(xyz, dtype=xyz.dtype, requires_grad=True, device="cuda") + 0
        screenspace_points.retain_grad()
        rs = GaussianRasterizationSettings(
            image_height=int(cam.height), image_width=int(cam.width), tanfovx=math.tan(cam.fovx * 0.5),
            tanfovy=math.tan(cam.fovy * 0.5), bg=bg, scale_modifier=1.0, z_near=g.z_near, z_far=g.z_far,
            use_sigmoid=g.use_sigmoid, sh_degree=g.active_sh_degree, campos=center, prefiltered=False, debug=False)
        img, depth, radii = GaussianRasterizer(raster_settings=rs)(
            means3D=xyz, means2D=screenspace_points, shs=g.get_features, colors_precomp=None,
            opacities=g.get_opacity, scales=g.get_scaling, rotations=g.get_rotation, cov3D_precomp=None,
            viewmatrix=view, projmatrix=proj)
        return img

    def step(gt, gt_ready=None):
        for p in params:
            p.grad = None
        nu = pt.sample_nu(cmm._nu[0], cmm.n_subframes)
        poses = pt.trajectory(cmm._trans._control_points[0], cmm._rot._control_points[0], nu,
                              ref_cam.projection_matrix)
        subframes = torch.stack([render(v, p, c, w["bg"]) for (v, p, c) in poses])   # scene/motion.py:141-145
        blurred = subframes.mean(dim=0)
        if gt_ready is not None:
            torch.cuda.current_stream().wait_event(gt_ready)
        loss = (blurred - gt).abs().mean()
        if lambda_t_smooth != 0.0:   # batchwise_smoothness_loss, utils/loss_utils.py:80-93
            loss = loss + lambda_t_smooth * (subframes[1:] - subframes[:-1]).abs().mean()
        loss.backward()
        return loss
    return step


# ------------------------------------------------------------------------------------------------
def workload_stats(w):
    """V, D, E, K, E_b of this rank's view (measurement only, outside the timed region)."""
    from deblurgs_b200 import _lib, rasterizer as rz
    lib = _lib.load()
    g, cmm, cam = w["gaussians"], w["cmm"], w["cam"]
    with torch.no_grad():
        view, proj, campos = cmm.get_trajectory_tensors(0)
        out = rz._forward_batched(g.get_xyz.detach(), g.get_features.detach(), None, g.get_opacity.detach(),
                                  g.get_scaling.detach(), g.get_rotation.detach(), None, view, proj, campos,
                                  w["bg"], cam.height, cam.width, cam.tanfovx, cam.tanfovy, 1.0, g.z_near,
                                  g.z_far, g.active_sh_degree, False, g.use_sigmoid, False, float(w["F"]))
        color, depth, radii, _, D, geom, binning, img = out
        stats = torch.zeros(3, dtype=torch.int64, device=color.device)
        rc = lib.dgs_debug_workload(_lib.ptr(geom), _lib.ptr(binning), _lib.ptr(img), w["P"], w["F"], cam.width,
                                    cam.height, D, _lib.ptr(stats),
                                    C.c_void_p(torch.cuda.current_stream().cuda_stream))
        _lib.check(rc, "dgs_debug_workload")
        E, K, Eb = (int(v) for v in stats.tolist())
        V = int((radii > 0).sum())
    return dict(V=V, D=int(D), E=E, K=K, E_b=Eb)


def algorithmic_bytes(w, st, sort_bits):
    """SURVEY.md 8(d) HBM byte model per blurry view, split per stage (the REFERENCE's algorithm: one 64-bit sort
    of D duplicates, 12-B pairs, one 8-bit pass per 8 key bits)."""
    P, F, W, H = w["P"], w["F"], w["W"], w["H"]
    M = w["scene"].shs.shape[1]
    G = 44 + 12 * M
    V, D = st["V"], st["D"]
    passes = math.ceil(sort_bits / 8)
    binning = 2 * 4 * P * F + (V * 16 + D * 12) + D * 12 * 2 * passes + D * 8   # scan + duplicate + sort + ranges
    return {
        "preprocess_fwd": P * G + V * 48,
        "binning": binning,
        "render_fwd": D * (4 + 44) + F * H * W * (16 + 8),
        "blur_mean": F * H * W * 12 + H * W * 12,
        "bwd_memset": V * 40,
        "render_bwd": D * (4 + 44) + F * H * W * (16 + 8) + V * 40,
        "preprocess_bwd": P * G + P * G + V * 40 + V * 48,
    }


def moved_bytes_binning(w, st, tile_key_bits):
    """Bytes THIS library's binning moves per blurry view (dgs_binning.cu): 4 depth-sort passes over the N entries
    (4-B keys read twice, 4-B values, 8 B written), the entry scan (8-B rectangle gather, 4 + 8 + 4 B written, 4 B
    read), and the tile sort (pass 1 generates its items and writes 8 B per duplicate; every later pass reads the
    4-B keys twice and the values once; the last pass writes only the 4-B Gaussian index)."""
    N, D = w["P"] * w["F"], st["D"]
    passes = max(1, math.ceil(tile_key_bits / 8))
    depth_sort = N * (4 + 8 + 8) * 4 - N * 4          # first pass has no value input
    scan = N * (4 + 8 + 4 + 8 + 4 + 4)
    gen_reads = 2 * N * 12                            # offsets + packed rectangles, read by the pass-1 up- and downsweep
    if passes == 1:
        tile = gen_reads + D * 4
    else:
        tile = gen_reads + D * 8 + (passes - 2) * D * (4 + 8 + 8) + D * (4 + 8 + 4)
    return depth_sort + scan + tile


def read_profile(lib):
    n = lib.dgs_profile_num_stages()
    ms = (C.c_double * n)()
    calls = (C.c_int64 * n)()
    rc = lib.dgs_profile_read(ms, calls, n, 1)
    if rc != 0:
        raise RuntimeError("dgs_profile_read failed")
    return {lib.dgs_profile_stage_name(i).decode(): (ms[i], calls[i]) for i in range(n)}


def cpu_baseline(bench_config):
    """PyTorch-CPU evaluation of the same path (oracle/raster_torch_cpu.py: test infrastructure, the checker) on all
    host cores: pose chain -> projection -> tile keys -> sort -> front-to-back composite -> mean -> L1 -> autograd
    backward.  Two bounded samples: (1) BASELINE.json's CPU-runnable config c1 in full (one whole blurry view,
    50 k Gaussians, 256x256, F=4); (2) ONE sub-frame of the benchmark's own workload, scaled to views/s by 1/F."""
    from deblurgs_b200 import synthetic
    from oracle import pose_torch as pt, raster_torch_cpu as rt
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)

    def setup(name):
        P, W, H, F, order = synthetic.get_config(name)
        cam = synthetic.make_camera(W, H)
        sc = synthetic.make_scene(P, cam, seed=0)
        tr = synthetic.make_trajectory(F, order, seed=1)
        params = [t.clone() for t in (sc.means3D, sc.scales, sc.rotations, sc.opacities, sc.shs)]
        return P, W, H, F, cam, tr, params, synthetic.make_background(), synthetic.make_target(cam, seed=2)

    # warm-up (thread pools, allocator) on the tiny config
    P, W, H, F, cam, tr, params, bg, gt = setup("tiny")
    rt.blurry_view_step(params, tr.ctrl_trans.clone(), tr.ctrl_rot.clone(), tr.nu, cam.projection_matrix_t(), bg, gt,
                        W, H, cam.tanfovx, cam.tanfovy)
    # (1) full c1 view
    P, W, H, F, cam, tr, params, bg, gt = setup("c1")
    t0 = time.perf_counter()
    rt.blurry_view_step(params, tr.ctrl_trans.clone(), tr.ctrl_rot.clone(), tr.nu, cam.projection_matrix_t(), bg, gt,
                        W, H, cam.tanfovx, cam.tanfovy)
    t_c1 = time.perf_counter() - t0
    # (2) one sub-frame of the benchmark workload, forward + backward
    P, W, H, F, cam, tr, params, bg, gt = setup(bench_config)
    for t in params:
        t.requires_grad_(True)
    v, p, c = pt.trajectory(tr.ctrl_trans, tr.ctrl_rot, tr.nu, cam.projection_matrix_t())[0]
    t0 = time.perf_counter()
    img = rt.render_view(*params, 3, v.float(), p.float(), c.float(), bg, W, H, cam.tanfovx, cam.tanfovy)[0]
    ((img - gt).abs().mean() / F).backward()
    t_sub = time.perf_counter() - t0
    return {"value": 1.0 / (t_sub * F), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "PyTorch-CPU (autograd, %d threads): one of the %d sub-frames of %s, forward + backward, in "
                      "%.1f s; views/s = 1 / (F x that)" % (cores, F, bench_config, t_sub),
            "c1_full": {"value": 1.0 / t_c1, "unit": UNIT,
                        "sample": "one whole c1 blurry view (50 k Gaussians, 256x256, F=4, cubic Bezier), forward + "
                                  "backward incl. the pose chain, in %.1f s" % t_c1}}


PARAM_NAMES = ["xyz", "features_dc", "features_rest", "scaling", "rotation", "opacity", "ctrl_trans", "ctrl_rot", "nu"]
DUMP_MAX_ELEMENTS = 1 << 20     # per array: 4 MB of float32, so that the nine gradients and the loss stay under 64 MB


def dump_outputs(w, loss, out_dir):
    """Writes what one step hands its caller -- the loss and the gradient of every parameter -- as <name>.npy (float32;
    the loss float64).  An array of more than DUMP_MAX_ELEMENTS elements is replaced by the elements at a fixed set of
    flat indices (seeded by its size, sorted), so two builds dumped with the same arguments compare element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([float(loss.item())], dtype=np.float64))
    params = w["gaussians"].parameters() + w["cmm"].parameters()
    for name, p in zip(PARAM_NAMES, params):
        g = p.grad.detach().reshape(-1).float()
        if g.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randperm(g.numel(), generator=torch.Generator().manual_seed(g.numel()))[:DUMP_MAX_ELEMENTS]
            g = g[idx.sort().values.to(g.device)]
        np.save(os.path.join(out_dir, name + ".npy"), g.cpu().numpy())


def time_steps(step, gt_dev, steps, world, device):
    """`steps` steps between two CUDA events on the current stream; ms per step, max over ranks."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(world)
    e0.record()
    for _ in range(steps):
        loss = step(gt_dev)
    e1.record()
    barrier(world)
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()) / steps, loss


def other_config(name, rank, world, device, steps=3, warmup=3):
    """BASELINE.json configs 3 and 4 in the same run: c3 = one 1080p view, its sub-frames sharded over the ranks (strong
    scaling: value = views/s of that one view); c4 = one 3 M-Gaussian view per rank (weak: value = world x views/s)."""
    strong = name == "c3"
    w = build_workload(name, 0 if strong else rank, device)
    if name == "c1":      # BASELINE config 1 (the CPU-runnable case): launch-bound kernel by kernel, so replayed as a graph
        step = make_step_ours(w, 1, 0.0, True)
    else:
        # graph replay everywhere (DGS_BENCH_EAGER_OTHERS=1: kernel by kernel, for comparison)
        gmode = os.environ.get("DGS_BENCH_EAGER_OTHERS") != "1"
        step = (make_step_subframe_sharded(w, world, gmode) if (strong and world > 1)
                else make_step_ours(w, 1 if strong else world, 0.0, gmode))
    mode = ("subframes-sharded-%d (NCCL all-reduce of the blurred image; gradient all-reduce overlapped with the backward)"
            % world) if (strong and world > 1) else None
    gt = w["gt_host"].to(device)
    for _ in range(warmup):
        step(gt)
    ms = time_steps(step, gt, steps, world, device)[0]
    loss = float(step(gt).item())
    P, W, H, F = w["P"], w["W"], w["H"], w["F"]
    mode_str = getattr(step, "mode", "kernel by kernel")
    del w, step
    torch.cuda.empty_cache()
    return {"workload": "%s: %d Gaussians, %dx%d, num_subframes=%d" % (name, P, W, H, F),
            "parallelism": mode if mode else ("single GPU" if (strong or name == "c1") else "views-dp%d" % world),
            "launch_mode": mode_str,
            "scaling": "strong" if strong else "weak", "steps": steps, "warmup": warmup, "ms_per_step": ms,
            "value": (1.0 if strong else world) * 1000.0 / ms, "unit": UNIT, "loss_last": loss}


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="c2")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--loss", default="l1", choices=["l1", "smooth"],
                    help="l1: mean|blur - gt| (headline); smooth: + 1e-3 * temporal smoothness of the sub-frames "
                         "(SURVEY 8d's second variant: non-uniform per-sub-frame gradients)")
    ap.add_argument("--split", default="views", choices=["views", "subframes"],
                    help="N > 1: views = one view per rank (weak scaling, headline); subframes = ONE view, its "
                         "sub-frames sharded over the ranks (strong scaling)")
    ap.add_argument("--no-graph", action="store_true", help="launch the step kernel by kernel instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the c3 / c4 lines")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and parameter gradients to DIR/<name>.npy "
                         "(a fixed sample of 2^20 elements of a larger gradient)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE JSON line: everything else any library prints while the run lasts (NCCL's version
    # banner, torch warnings) goes to stderr at the file-descriptor level; `emit` writes to the real stdout.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    rank, world, local = dist_setup(args.gpus)
    if args.impl == "reference" and rank != 0:
        return   # the reference is single-GPU: rank 0 alone runs it
    device = torch.device("cuda", local)
    eff_world = 1 if args.impl == "reference" else world
    sharded = args.impl == "ours" and args.split == "subframes" and eff_world > 1
    w = build_workload(args.config, 0 if sharded else rank, device)
    F = w["F"]
    lam = 1e-3 if args.loss == "smooth" else 0.0
    use_graph = args.impl == "ours" and not args.no_graph

    if args.impl == "ours":
        from deblurgs_b200 import _lib
        lib = _lib.load()
        step = make_step_subframe_sharded(w, eff_world, use_graph) if sharded else make_step_ours(w, eff_world, lam, use_graph)
    else:
        lib = None
        if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "diff_gaussian_rasterization")):
            emit({"impl": "reference", "unavailable": "baseline/_ref is not installed"})
            return
        step = make_step_reference(w, lam)

    gt_dev = w["gt_host"].to(device)
    for _ in range(args.warmup):
        step(gt_dev)
    barrier(eff_world)

    # ---- device-resident timing: inputs already in HBM, CUDA events, max over ranks
    if lib is not None:
        lib.dgs_launch_count(1)
    sampler = ClockSampler(local)
    sampler.start()
    ms_step, last_loss = time_steps(step, gt_dev, args.steps, eff_world, device)
    sampler.stop_flag = True
    sampler.join()
    launches = None
    if lib is not None:
        launches = int(lib.dgs_launch_count(0))
        if step.graph is not None:     # kernels inside a replayed graph are not seen by the launch counter
            step.graph.check()
            launches += step.graph.launches_per_replay * args.steps
    if args.dump_outputs and rank == 0:   # after check(): a replay past the graph's capacity is redone there
        dump_outputs(w, step.graph.loss if getattr(step, "graph", None) is not None else last_loss, args.dump_outputs)
    views_per_step = 1 if sharded else eff_world
    value = views_per_step * 1000.0 / ms_step

    # ---- end to end through the public API: pinned-host ground truth in, loss scalar out, every step
    # (the upload runs on a side stream into one of two preallocated device buffers, as a data loader's
    # prefetch would, and is awaited before the loss; the loss read-back makes every step synchronous)
    barrier(eff_world)
    copy_stream = torch.cuda.Stream(device)
    gt_bufs = [torch.empty_like(gt_dev), torch.empty_like(gt_dev)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    t_prev, step_wall = t0, []
    for k in range(args.steps):
        gt = gt_bufs[k & 1]
        with torch.cuda.stream(copy_stream):
            gt.copy_(w["gt_host"], non_blocking=True)
            gt_ready = copy_stream.record_event()
        loss = step(gt, gt_ready)
        loss_host = loss.item()
        # capacity exceeded: re-captured + replayed (with collectives inside the graph the check is itself a collective:
        # done once after the loop instead; the scene does not change here)
        if getattr(step, "graph", None) is not None and eff_world == 1 and step.graph.check():
            loss_host = step.graph.loss.item()
        t_now = time.perf_counter()
        step_wall.append((t_now - t_prev) * 1e3)
        t_prev = t_now
    torch.cuda.synchronize()
    t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=device)
    if eff_world > 1:
        import torch.distributed as dist
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = views_per_step * args.steps / float(t_e2e.item())

    # ---- per-stage CUDA-event times: a separate pass, kernel by kernel (events inside a replayed graph cannot be read)
    prof = None
    if lib is not None and not sharded:
        w["gaussians"].grad_sink = None
        eager = make_step_ours(w, 1, lam, False)
        for p in w["gaussians"].parameters():
            p.grad = None
        for _ in range(2):
            eager(gt_dev)
        torch.cuda.synchronize()
        lib.dgs_profile_read(None, None, 0, 1)
        lib.dgs_profile_enable(1)
        n_prof = 5
        for _ in range(n_prof):
            eager(gt_dev)
        torch.cuda.synchronize()
        prof = read_profile(lib)
        lib.dgs_profile_enable(0)

    # ---- BASELINE.json's other shapes (c3 sub-frame split, c4 view batch) in the same run
    others = None
    if args.impl == "ours" and not args.no_other_configs and args.config == "c2" and not sharded:
        others = {}
        for name in (("c1",) if eff_world == 1 else ()) + ("c3", "c4"):
            try:
                others[name] = other_config(name, rank, eff_world, device)
            except Exception as e:   # never lose the headline line to an out-of-memory on the big shapes
                others[name] = {"error": "%s: %s" % (type(e).__name__, str(e)[:200])}
                torch.cuda.empty_cache()

    if eff_world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    clocks = sampler.summary()
    if sharded:
        par, scaling = "subframes-sharded-%d" % eff_world, "strong"
    else:
        par, scaling = "views-dp%d" % eff_world, "weak"
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": eff_world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_step, "ms_per_subframe": ms_step / F,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "%s: %d Gaussians, %dx%d, num_subframes=%d, SH degree 3, se3 Bezier order %d, "
                               "one blurry view per %s per step (fwd+bwd, %s), inputs larger than L2"
                               % (args.config, w["P"], w["W"], w["H"], F, w["order"], "job" if sharded else "GPU",
                                  "L1 loss" if lam == 0.0 else "L1 + 1e-3 temporal-smoothness loss"),
                   "parallelism": par},
        "loss_last": loss_host,
        "launch_mode": getattr(step, "mode", "kernel by kernel"),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(w["gt_host"].numel() * 4),
                "d2h_bytes_per_step": 4 + (24 if use_graph else 0),
                "ms_per_step_min_median_max": [round(min(step_wall), 3), round(statistics.median(step_wall), 3),
                                               round(max(step_wall), 3)]},
    }
    if others:
        out["other_configs"] = others
    if args.impl == "reference":
        out["impl"] = "reference"
        out["launch_mode"] = "kernel by kernel (the reference synchronises once per sub-frame)"
        out["reference_kind"] = ("reference CUDA extension (baseline/_ref, unmodified, sm_100 build) on the same "
                                 "B200, driven by the reference's per-sub-frame loop")
        out["cpu_baseline"] = {"value": value, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                               "sample": "full workload; the reference implementation of this path is itself a "
                                         "CUDA extension, so this arm runs on the GPU, host cores only drive it"}
        out["gpu_launches"] = 0
        emit(out)
        return

    out["gpu_launches"] = launches
    if prof is None:      # sub-frame-sharded run: no per-stage breakdown
        emit(out)
        return
    st = workload_stats(w)
    tb, sb = C.c_int(0), C.c_int(0)
    lib.dgs_key_bits(w["W"], w["H"], F, C.byref(tb), C.byref(sb))
    abytes = algorithmic_bytes(w, st, 32 + tb.value)       # the reference sorts [tile | depth] per sub-frame
    stage_ms = {k: (v[0] / n_prof) for k, v in prof.items() if v[1] > 0}          # ms per step
    stage_ms["binning"] = sum(stage_ms.get(k, 0.0) for k in ("depth_sort", "scan", "tile_sort"))
    out["stage_ms_per_step"] = {k: round(v, 4) for k, v in stage_ms.items()}
    out["stage_ms_note"] = "CUDA events around every stage in a separate kernel-by-kernel pass (5 steps)"
    out["workload_stats"] = st
    # FP32 FMA rate of this GPU, measured (register-resident FMA kernel) right here
    pk, mhz = C.c_double(0.0), C.c_double(0.0)
    _lib.check(lib.dgs_measure_fp32_peak(C.byref(pk), C.byref(mhz), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
               "dgs_measure_fp32_peak")
    fp32_peak = pk.value
    n_sm = torch.cuda.get_device_properties(device).multi_processor_count
    flops = {"render_fwd": 14 * st["E"] + 18 * st["K"], "render_bwd": 16 * st["E_b"] + 88 * st["K"]}
    # dominant kernel among the stages with an algorithmic work figure
    dom = max((k for k in stage_ms if k in flops or k in abytes), key=stage_ms.get)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    limiter = None
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f).get(args.config, {})
        traffic, limiter = tj.get(dom), tj.get("limiters", {}).get(dom)
    hbm, src = measured_peaks()
    if dom in flops:
        ach = flops[dom] / (stage_ms[dom] * 1e-3) / 1e12
        out["roofline"] = {"kernel": dom, "bound": "fp32", "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s",
                           "frac": ach / fp32_peak, "traffic": traffic,
                           "peak_source": "measured in this run: FP32 FMA kernel, best of 6 (implies %.0f MHz x %d SMs x 128 "
                                          "lanes x 2; the SM clock sampled during the timed region was %s MHz)"
                                          % (mhz.value, n_sm, clocks["sm_mhz"]),
                           "algorithmic_flops_per_launch": flops[dom], "ms_per_launch": stage_ms[dom]}
        if limiter:   # what ncu says binds the kernel (recorded from the committed capture, not measured in this run)
            out["roofline"]["measured_limiter"] = limiter
        if traffic:   # why the bound is not HBM: measured DRAM traffic of the same kernel against the copy bandwidth
            out["roofline"]["dram_gbs"] = traffic / (stage_ms[dom] * 1e-3) / 1e9
            out["roofline"]["dram_frac_of_hbm_peak"] = out["roofline"]["dram_gbs"] / hbm
    else:
        ach = abytes[dom] / (stage_ms[dom] * 1e-3) / 1e9
        out["roofline"] = {"kernel": dom, "bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s",
                           "frac": ach / hbm, "traffic": traffic, "peak_source": src,
                           "algorithmic_bytes_per_launch": abytes[dom], "ms_per_launch": stage_ms[dom]}
    # the HBM-bound stages: SURVEY 8(d)'s algorithmic bytes (the reference's algorithm) next to the bytes this
    # library's own binning actually moves
    hbm_stages = ["preprocess_fwd", "binning", "bwd_memset", "preprocess_bwd"]
    hb = sum(abytes[k] for k in hbm_stages if k in stage_ms)
    ht = sum(stage_ms[k] for k in hbm_stages if k in stage_ms)
    moved = moved_bytes_binning(w, st, max(1, (w["cam"].width + 15) // 16 * ((w["cam"].height + 15) // 16) - 1).bit_length())
    out["roofline_hbm_group"] = {
        "kernels": hbm_stages, "bound": "hbm", "achieved": hb / (ht * 1e-3) / 1e9, "peak": hbm, "unit": "GB/s",
        "frac": hb / (ht * 1e-3) / 1e9 / hbm, "peak_source": src, "algorithmic_bytes": hb, "ms": ht,
        "binning": {"ms": stage_ms["binning"], "algorithmic_bytes": abytes["binning"],
                    "algorithmic_gbs": abytes["binning"] / (stage_ms["binning"] * 1e-3) / 1e9,
                    "moved_bytes": moved, "moved_gbs": moved / (stage_ms["binning"] * 1e-3) / 1e9,
                    "moved_frac_of_hbm_peak": moved / (stage_ms["binning"] * 1e-3) / 1e9 / hbm,
                    "note": "algorithmic = the reference's scan + duplicateWithKeys + one 64-bit sort of 12-B pairs + "
                            "identifyTileRanges (SURVEY 8d); moved = what dgs_binning.cu reads and writes"}}
    if not args.no_cpu_baseline and eff_world == 1:
        out["cpu_baseline"] = cpu_baseline(args.config)
    emit(out)


if __name__ == "__main__":
    main()
