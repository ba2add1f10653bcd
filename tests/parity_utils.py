"""Shared helpers for the GPU parity tests: run libdgs_b200 (through the package's C-ABI binding), decode
every intermediate the reference defines, and compare them with the reference's outputs stored in
tests/golden/parity.npz."""
import ctypes as C
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from deblurgs_b200 import _lib, synthetic  # noqa: E402
from deblurgs_b200 import rasterizer as rz  # noqa: E402
from deblurgs_b200.pose import bezier_se3_poses  # noqa: E402


def make_inputs(name, device="cuda", sh_degree=3, P=None, F=None):
    Pn, W, H, Fn, Cn = synthetic.CONFIGS[name]
    P = Pn if P is None else P
    F = Fn if F is None else F
    cam = synthetic.make_camera(W, H)
    scene = synthetic.make_scene(P, cam, sh_degree=sh_degree).to(device)
    traj = synthetic.make_trajectory(F, Cn).to(device)
    bg = synthetic.make_background().to(device)
    view, proj, campos = bezier_se3_poses(traj.ctrl_trans, traj.ctrl_rot, traj.nu,
                                          cam.projection_matrix_t().to(device))
    return cam, scene, traj, bg, view.contiguous(), proj.contiguous(), campos.contiguous()


def ours_forward(cam, scene, bg, view, proj, campos, sh_degree=None, use_sigmoid=False, colors_precomp=None,
                 cov3D_precomp=None, scale_modifier=1.0, want_blur=True, exact=False):
    sh_degree = scene.sh_degree if sh_degree is None else sh_degree
    shs = None if colors_precomp is not None else scene.shs
    scales = None if cov3D_precomp is not None else scene.scales
    rots = None if cov3D_precomp is not None else scene.rotations
    out = rz._forward_batched(scene.means3D, shs, colors_precomp, scene.opacities, scales, rots, cov3D_precomp,
                              view, proj, campos, bg, cam.height, cam.width, cam.tanfovx, cam.tanfovy,
                              scale_modifier, 0.2, 100.0, sh_degree, False, use_sigmoid, want_blur,
                              float(view.shape[0]), exact=exact)
    color, depth, radii, blur, D, geom, binning, img = out
    return dict(color=color, depth=depth, radii=radii, blur=blur, num_rendered=D, geom=geom, binning=binning,
                img=img)


def ours_decode(fw, P, F, W, H):
    lib = _lib.load()
    dev = fw["color"].device
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    N = P * F
    D = fw["num_rendered"]
    tiles = ((W + 15) // 16) * ((H + 15) // 16)
    f32 = dict(dtype=torch.float32, device=dev)
    i32 = dict(dtype=torch.int32, device=dev)
    d = dict(depths=torch.zeros((F, P), **f32), means2D=torch.zeros((F, P, 2), **f32),
             conic_opacity=torch.zeros((F, P, 4), **f32), rgb=torch.zeros((F, P, 3), **f32),
             clamped=torch.zeros((F, P, 3), **f32), tiles_touched=torch.zeros((F, P), **i32),
             point_offsets=torch.zeros((F, P), **i32),
             keys=torch.zeros(D, dtype=torch.int64, device=dev), point_list=torch.zeros(D, **i32),
             ranges=torch.zeros((F, tiles, 2), **i32), final_T=torch.zeros((F, H, W), **f32),
             n_contrib=torch.zeros((F, H, W), **i32))
    p = _lib.ptr
    if N:
        _lib.check(lib.dgs_debug_geometry(p(fw["geom"]), P, F, p(d["depths"]), p(d["means2D"]),
                                          p(d["conic_opacity"]), p(d["rgb"]), p(d["clamped"]),
                                          p(d["tiles_touched"]), p(d["point_offsets"]), st), "debug_geometry")
    if N:
        _lib.check(lib.dgs_debug_binning(p(fw["geom"]), p(fw["binning"]), p(fw["img"]), P, F, W, H, D, p(d["keys"]),
                                         p(d["point_list"]), p(d["ranges"]), st), "debug_binning")
    _lib.check(lib.dgs_debug_image(p(fw["img"]), F, W, H, p(d["final_T"]), p(d["n_contrib"]), st), "debug_image")
    tb, sb = C.c_int(0), C.c_int(0)
    lib.dgs_key_bits(W, H, F, C.byref(tb), C.byref(sb))
    d["tile_bits"], d["subframe_bits"] = tb.value, sb.value
    torch.cuda.synchronize(dev)
    return d


def ours_backward(cam, scene, bg, view, proj, campos, fw, dL_dpix, dL_ddepth, sh_degree=None, use_sigmoid=False,
                  colors_precomp=None, cov3D_precomp=None, scale_modifier=1.0):
    sh_degree = scene.sh_degree if sh_degree is None else sh_degree
    P, F = scene.means3D.shape[0], view.shape[0]
    shs = None if colors_precomp is not None else scene.shs
    scales = None if cov3D_precomp is not None else scene.scales
    rots = None if cov3D_precomp is not None else scene.rotations
    M = shs.shape[1] if shs is not None else 0
    names = ["dL_dmeans2D", "dL_dmeans3D", "dL_dsh", "dL_dopacity", "dL_dscales", "dL_drotations", "dL_dcolors",
             "dL_dcov3D", "dL_dviewmatrix", "dL_dprojmatrix"]
    out = rz._backward_batched(P, F, M, fw["num_rendered"], scene.means3D, shs, colors_precomp, scene.opacities,
                               scales, rots, cov3D_precomp, view, proj, campos, bg, cam.height, cam.width,
                               cam.tanfovx, cam.tanfovy, scale_modifier, 0.2, 100.0, sh_degree, use_sigmoid,
                               fw["radii"], fw["geom"], fw["binning"], fw["img"], dL_dpix, dL_ddepth, True,
                               want_stats=True)
    return dict(zip(names + ["densify_stats"], out))


GOLDEN = os.path.join(ROOT, "tests", "golden", "parity.npz")
WHOLE = 384       # float tensors up to this size are stored whole
SAMPLE = 320      # larger ones: this many elements at seeded random positions ...
TAIL = 64         # ... and their last elements (the last Gaussians; the last rows of the last image)
_STORE = None


def _sample_index(n):
    if n <= WHOLE:
        return torch.arange(n)
    idx = torch.randint(0, n - TAIL, (SAMPLE,), generator=torch.Generator().manual_seed(n))
    return torch.cat([idx.unique(), torch.arange(n - TAIL, n)])


class Golden:
    """Stored outputs of one test case, in tests/golden/parity.npz as three arrays per case: <case>.names (the fields),
    <case>.exact (per bit-exact field: the SHA-256 digest of its bytes, then its shape as four int64) and
    <case>.sample (per float field, concatenated: the tensor whole up to WHOLE elements, otherwise the elements at
    _sample_index, each followed by the tensor's max |x|).

    The vectors were recorded from this library's kernels as they were when the parity suite last ran against the
    reference's own CUDA rasterizer, simple-knn and extension module on a B200, with every list bit-identical and every
    image and gradient within the bars the tests apply (profiles/r2_final_gpu_tests.log): they stand in for the
    reference's outputs, which need the reference's sources to produce.
    With DGS_RECORD_GOLDEN=<dir> set, the tests write one <case>.npz per case to <dir> instead of comparing;
    pack(<dir>) merges them into tests/golden/parity.npz."""

    def __init__(self, case):
        global _STORE
        self.case = case
        self.record_dir = os.environ.get("DGS_RECORD_GOLDEN")
        self.exacts, self.samples = {}, {}
        if self.record_dir:
            return
        if _STORE is None:
            with np.load(GOLDEN) as z:
                _STORE = {k: z[k] for k in z.files}
        names = list(_STORE[case + ".names"])
        ex, sm = _STORE[case + ".exact"], _STORE[case + ".sample"]
        off = 0
        for name in names:
            kind, key = name.split(":", 1)
            if kind == "x":
                self.exacts[key] = ex[len(self.exacts)]
            else:
                n = int(kind[1:])
                self.samples[key] = sm[off:off + n + 1]
                off += n + 1

    def exact(self, key, t):
        """t bit for bit."""
        t = t.detach().contiguous().cpu()
        assert t.dim() <= 4
        shape = np.zeros(4, np.int64)
        shape[:t.dim()] = t.shape
        d = np.concatenate([np.frombuffer(hashlib.sha256(t.view(torch.uint8).numpy().tobytes()).digest(), np.uint8),
                            shape.view(np.uint8)])
        if self.record_dir:
            self.exacts[key] = d
        assert np.array_equal(self.exacts[key], d), (self.case, key, tuple(t.shape))

    def sample(self, key, t):
        """(this run's sample of t, the stored sample, the stored max |x| of the whole tensor), float64 on the CPU."""
        t = t.detach().reshape(-1)
        n = t.numel()
        mine = t[_sample_index(n).to(t.device)].cpu()
        if self.record_dir:
            self.samples[key] = np.append(mine.float().numpy(), np.float32(t.abs().max().item() if n else 0.0))
        stored = torch.from_numpy(self.samples[key]).double()
        assert stored.numel() == mine.numel() + 1, (self.case, key)
        return mine.double(), stored[:-1], float(stored[-1])

    def abs_close(self, key, t, tol):
        """max |t - stored| <= tol on the stored elements."""
        a, b, _ = self.sample(key, t)
        err = float((a - b).abs().max()) if a.numel() else 0.0
        assert err <= tol, (self.case, key, err, tol)

    def rel_close(self, key, t, tol):
        """max |t - stored| / max |stored| <= tol (the stored elements' errors over the whole tensor's max)."""
        a, b, m = self.sample(key, t)
        err = float((a - b).abs().max()) / max(m, 1e-30) if a.numel() else 0.0
        assert err <= tol, (self.case, key, err, tol)

    def rel_err(self, key, t, floor_frac=1e-3):
        """rel_err (below) of t against the stored elements."""
        a, b, m = self.sample(key, t)
        if m == 0:
            return float((a - b).abs().max()) if a.numel() else 0.0
        return float(((a - b).abs() / b.abs().clamp_min(floor_frac * m)).max())

    def done(self):
        if not self.record_dir:
            return
        names = ["x:" + k for k in self.exacts] + ["s%d:%s" % (len(v) - 1, k) for k, v in self.samples.items()]
        ex = np.stack(list(self.exacts.values())) if self.exacts else np.zeros((0, 64), np.uint8)
        sm = np.concatenate(list(self.samples.values())) if self.samples else np.zeros(0, np.float32)
        os.makedirs(self.record_dir, exist_ok=True)
        np.savez_compressed(os.path.join(self.record_dir, self.case + ".npz"), names=np.array(names), exact=ex,
                            sample=sm.astype(np.float32))


def pack(record_dir, out=GOLDEN):
    """Merge the per-case files a recording run wrote into one archive."""
    arrays = {}
    for f in sorted(os.listdir(record_dir)):
        with np.load(os.path.join(record_dir, f)) as z:
            for k in z.files:
                arrays[f[:-len(".npz")] + "." + k] = z[k]
    np.savez_compressed(out, **arrays)


def rel_err(a, b, floor_frac=1e-3):
    """max |a-b| / max(|b|, floor) with floor = floor_frac * max|b| (relative error that does not blow
    up on entries that are ~0 by cancellation)."""
    a, b = a.double(), b.double()
    scale = b.abs().max().item()
    if scale == 0:
        return (a - b).abs().max().item()
    denom = torch.clamp(b.abs(), min=floor_frac * scale)
    return ((a - b).abs() / denom).max().item()
