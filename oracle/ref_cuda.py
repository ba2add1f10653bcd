"""TEST INFRASTRUCTURE ONLY -- never imported by the product (deblurgs_b200/).

ctypes driver for oracle/_ref/libref_dgr.so: the reference's own CUDA rasterizer and simple-knn
compiled in place from /root/reference by oracle/Makefile, behind the C shim oracle/ref_shim.cu.
It lets the GPU parity tests run the *reference implementation itself* on exactly the device
buffers handed to libdgs_b200.so, and decodes the reference's opaque state buffers
(GeometryState / BinningState / ImageState, cuda_rasterizer/rasterizer_impl.h:31-63,
rasterizer_impl.cu:155-194) into named tensors.
"""
import ctypes as C
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_ref", "libref_dgr.so")
_ALLOC = C.CFUNCTYPE(C.c_void_p, C.c_size_t)
_lib = None


def available():
    return os.path.exists(LIB_PATH)


def load():
    global _lib
    if _lib is None:
        lib = C.CDLL(LIB_PATH)
        p, i, f = C.c_void_p, C.c_int, C.c_float
        lib.ref_forward.restype = i
        lib.ref_forward.argtypes = [_ALLOC, _ALLOC, _ALLOC, i, i, i, p, i, i, p, p, p, p, p, f, p, p, p, p, p,
                                    f, f, f, f, i, p, p, p, i]
        lib.ref_backward.restype = None
        lib.ref_backward.argtypes = [i, i, i, i, p, i, i, p, p, p, p, f, p, p, p, p, p, f, f, f, f, p, p, p, p,
                                     p, p] + [p] * 12 + [i]
        lib.ref_knn.restype = None
        lib.ref_knn.argtypes = [i, p, p]
        lib.ref_sync.restype = i
        _lib = lib
    return _lib


def _ptr(t):
    return None if (t is None or t.numel() == 0) else t.data_ptr()


class _Buf:
    def __init__(self, device):
        self.device = device
        self.t = torch.empty(0, dtype=torch.uint8, device=device)
        self.cb = _ALLOC(self._alloc)

    def _alloc(self, n):
        self.t = torch.zeros(int(n), dtype=torch.uint8, device=self.device)
        return self.t.data_ptr()


def _align(x, a=128):
    return (x + a - 1) // a * a


def _carve(buf, specs):
    """specs: list of (name, dtype, count). Mirrors `obtain` (128-B alignment on the absolute address)."""
    base = buf.data_ptr()
    off = 0
    out = {}
    for name, dtype, count in specs:
        off = _align(base + off) - base
        nbytes = count * torch.empty(0, dtype=dtype).element_size()
        out[name] = buf[off:off + nbytes].view(dtype)
        off += nbytes
    return out


def forward(means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, viewmatrix, projmatrix,
            campos, bg, W, H, tanfovx, tanfovy, sh_degree, scale_modifier=1.0, z_near=0.2, z_far=100.0,
            prefiltered=False, use_sigmoid=False):
    """One reference forward (single view). All tensors CUDA fp32 contiguous. The reference launches on
    the legacy default stream; callers must be on torch's default stream."""
    lib = load()
    dev = means3D.device
    P = means3D.shape[0]
    M = shs.shape[1] if shs is not None and shs.numel() else 0
    color = torch.zeros((3, H, W), dtype=torch.float32, device=dev)
    depth = torch.zeros((1, H, W), dtype=torch.float32, device=dev)
    radii = torch.zeros(P, dtype=torch.int32, device=dev)
    geom, binning, img = _Buf(dev), _Buf(dev), _Buf(dev)
    torch.cuda.synchronize(dev)
    R = lib.ref_forward(geom.cb, binning.cb, img.cb, P, sh_degree, M, _ptr(bg), W, H, _ptr(means3D), _ptr(shs),
                        _ptr(colors_precomp), _ptr(opacities), _ptr(scales), scale_modifier, _ptr(rotations),
                        _ptr(cov3D_precomp), _ptr(viewmatrix), _ptr(projmatrix), _ptr(campos), tanfovx, tanfovy,
                        z_near, z_far, int(prefiltered), _ptr(color), _ptr(depth), _ptr(radii), int(use_sigmoid))
    lib.ref_sync()
    g = _carve(geom.t, [("depths", torch.float32, P), ("pre_sigmoid", torch.float32, 3 * P),
                        ("internal_radii", torch.int32, P), ("means2D", torch.float32, 2 * P),
                        ("cov3D", torch.float32, 6 * P), ("conic_opacity", torch.float32, 4 * P),
                        ("rgb", torch.float32, 3 * P), ("tiles_touched", torch.int32, P)])
    b = _carve(binning.t, [("point_list", torch.int32, R), ("point_list_unsorted", torch.int32, R),
                           ("point_list_keys", torch.int64, R), ("point_list_keys_unsorted", torch.int64, R)])
    N = W * H
    im = _carve(img.t, [("accum_alpha", torch.float32, N), ("n_contrib", torch.int32, N),
                        ("ranges", torch.int32, 2 * N)])
    return dict(color=color, depth=depth, radii=radii, num_rendered=R, geom_buf=geom.t, binning_buf=binning.t,
                img_buf=img.t, geom=g, binning=b, image=im)


def backward(fw, means3D, shs, colors_precomp, scales, rotations, cov3D_precomp, viewmatrix, projmatrix, campos,
             bg, W, H, tanfovx, tanfovy, sh_degree, dL_dpix, dL_dpixdepth, scale_modifier=1.0, z_near=0.2,
             z_far=100.0, use_sigmoid=False):
    """Reference backward for a forward result `fw` (dict from forward()). Returns the 12 gradient tensors
    the reference binding allocates (rasterize_points.cu:163-175)."""
    lib = load()
    dev = means3D.device
    P = means3D.shape[0]
    M = shs.shape[1] if shs is not None and shs.numel() else 0
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    out = dict(dL_dmeans3D=z(P, 3), dL_dmeans2D=z(P, 3), dL_dcolors=z(P, 3), dL_dconic=z(P, 2, 2),
               dL_dopacity=z(P, 1), dL_dcov3D=z(P, 6), dL_dsh=z(P, M, 3), dL_dscales=z(P, 3),
               dL_drotations=z(P, 4), dL_ddepths=z(P, 1), dL_dviewmatrix=z(4, 4), dL_dprojmatrix=z(4, 4))
    torch.cuda.synchronize(dev)
    lib.ref_backward(P, sh_degree, M, fw["num_rendered"], _ptr(bg), W, H, _ptr(means3D), _ptr(shs),
                     _ptr(colors_precomp), _ptr(scales), scale_modifier, _ptr(rotations), _ptr(cov3D_precomp),
                     _ptr(viewmatrix), _ptr(projmatrix), _ptr(campos), tanfovx, tanfovy, z_near, z_far,
                     _ptr(fw["radii"]), _ptr(fw["geom_buf"]), _ptr(fw["binning_buf"]), _ptr(fw["img_buf"]),
                     _ptr(dL_dpix), _ptr(dL_dpixdepth),
                     _ptr(out["dL_dmeans2D"]), _ptr(out["dL_dconic"]), _ptr(out["dL_dopacity"]),
                     _ptr(out["dL_dcolors"]), _ptr(out["dL_dmeans3D"]), _ptr(out["dL_dcov3D"]), _ptr(out["dL_dsh"]),
                     _ptr(out["dL_dscales"]), _ptr(out["dL_drotations"]), _ptr(out["dL_ddepths"]),
                     _ptr(out["dL_dviewmatrix"]), _ptr(out["dL_dprojmatrix"]), int(use_sigmoid))
    lib.ref_sync()
    return out


def knn(points):
    lib = load()
    pts = points.float().contiguous()
    out = torch.zeros(pts.shape[0], dtype=torch.float32, device=pts.device)
    torch.cuda.synchronize(pts.device)
    lib.ref_knn(pts.shape[0], _ptr(pts), _ptr(out))
    lib.ref_sync()
    return out


TRUTH_LIB_PATH = os.path.join(HERE, "_build", "libtruth_bwd.so")
_truth = None


def truth_blend_backward(W, H, ranges, point_list, means2D, conic_opacity, rgb, depths, n_contrib, bg, dL_dpix,
                         dL_dpixdepth, z_far=100.0):
    """Float64 evaluation of the tile-blend backward (oracle/truth_bwd.cu, built by `make -C oracle truth`) on the
    forward state of one view: ranges [tiles, 2] and point_list of that view's tile lists, the per-Gaussian means2D,
    conic_opacity, rgb and depths, the per-pixel n_contrib (the decoded GeometryState / BinningState / ImageState
    arrays).  Same blend decisions as the float forward, float64 values and sums. Returns the tuple
    rn.preprocess_backward takes: (dL_dmean2D [P,2] w.r.t. NDC, dL_dconic [P,3], dL_dopacity [P], dL_dcolor [P,3],
    dL_ddepth [P]) as float64 CUDA tensors."""
    global _truth
    if _truth is None:
        lib = C.CDLL(TRUTH_LIB_PATH)
        lib.truth_blend_backward.restype = None
        lib.truth_blend_backward.argtypes = [C.c_int, C.c_int] + [C.c_void_p] * 8 + [C.c_float] + [C.c_void_p] * 7
        _truth = lib
    dev = bg.device
    P = means2D.shape[0]
    z = lambda *s: torch.zeros(s, dtype=torch.float64, device=dev)
    dmean, dconic, dop, dcol, ddep = z(P, 2), z(P, 3), z(P), z(P, 3), z(P)
    args = [t.contiguous() for t in (ranges, point_list, means2D, conic_opacity, rgb, depths, n_contrib, bg)]
    grads = [t.contiguous() for t in (dL_dpix, dL_dpixdepth)]
    torch.cuda.synchronize(dev)
    _truth.truth_blend_backward(W, H, *[_ptr(t) for t in args], z_far, *[_ptr(t) for t in grads], _ptr(dmean),
                                _ptr(dconic), _ptr(dop), _ptr(dcol), _ptr(ddep))   # legacy default stream
    torch.cuda.synchronize(dev)
    return dmean, dconic, dop, dcol, ddep
