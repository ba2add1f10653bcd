"""ctypes binding of libdgs_b200.so (the C-ABI declared in include/dgs_b200.h).

There is no fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DGS_B200_LIB: another build of the same library (A/B measurements of kernel variants); the default is the in-tree build
LIB_PATH = os.environ.get("DGS_B200_LIB") or os.path.join(_HERE, "libdgs_b200.so")

ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_size_t)

_p = C.c_void_p
_i = C.c_int
_f = C.c_float
_i64 = C.c_int64

_FWD_COMMON = [_p, _i, _i,                    # background, width, height
               _p, _p, _p,                    # means3D, shs, colors_precomp
               _p, _p, _f,                    # opacities, scales, scale_modifier
               _p, _p,                        # rotations, cov3D_precomp
               _p, _p, _p,                    # view, proj, campos
               _f, _f, _f, _f]                # tanfovx, tanfovy, z_near, z_far

SIGNATURES = {
    "dgs_last_error": (C.c_char_p, []),
    "dgs_version": (_i, []),
    "dgs_compiled_arch": (_i, []),
    "dgs_key_bits": (_i, [_i, _i, _i, C.POINTER(_i), C.POINTER(_i)]),
    "dgs_blur_forward": (_i, [ALLOC_FN, _p, ALLOC_FN, _p, ALLOC_FN, _p,
                              _i, _i, _i, _i] + _FWD_COMMON +
                         [_i, _i, _p, _p, _p, _p, _f, C.POINTER(_i64), _p]),
    "dgs_blur_forward_hint": (_i, [ALLOC_FN, _p, ALLOC_FN, _p, ALLOC_FN, _p,
                                   _i, _i, _i, _i] + _FWD_COMMON +
                              [_i, _i, _p, _p, _p, _p, _f, _i64, C.POINTER(_i64), _p]),
    "dgs_blur_forward_aa": (_i, [ALLOC_FN, _p, ALLOC_FN, _p, ALLOC_FN, _p,
                                 _i, _i, _i, _i] + _FWD_COMMON +
                            [_i, _i, _p, _p, _p, _p, _f, _i64, C.POINTER(_i64), _i, _p]),
    "dgs_blur_forward_contrib": (_i, [ALLOC_FN, _p, ALLOC_FN, _p, ALLOC_FN, _p,
                                      _i, _i, _i, _i] + _FWD_COMMON +
                                 [_i, _i, _p, _p, _p, _p, _f, _i64, C.POINTER(_i64), _i, _p, _p, _p]),
    "dgs_blur_forward_status": (_i, [_p, _i, _i, C.POINTER(_i64), C.POINTER(_i), _p]),
    "dgs_blur_forward_status_offset": (C.c_size_t, [_i, _i]),
    "dgs_blur_backward_scratch_bytes": (C.c_size_t, [_i, _i]),
    "dgs_blur_backward": (_i, [_i, _i, _i, _i, _i64] + _FWD_COMMON +
                          [_i, _p, _p, _p, _p, _p, _p, _p, _f, _p] + [_p] * 11 + [_p]),
    "dgs_blur_backward_range": (_i, [_i, _i, _i, _i, _i64] + _FWD_COMMON +
                                [_i, _p, _p, _p, _p, _p, _p, _p, _f, _p] + [_p] * 11 + [_i64, _i64, _i, _p]),
    "dgs_blur_backward_range_aa": (_i, [_i, _i, _i, _i, _i64] + _FWD_COMMON +
                                   [_i, _p, _p, _p, _p, _p, _p, _p, _f, _p] + [_p] * 11 + [_i64, _i64, _i, _i, _p]),
    "dgs_forward": (_i, [ALLOC_FN, _p, ALLOC_FN, _p, ALLOC_FN, _p,
                         _i, _i, _i] + _FWD_COMMON + [_i, _i, _p, _p, _p, C.POINTER(_i64), _p]),
    "dgs_backward": (_i, [_i, _i, _i, _i64] + _FWD_COMMON +
                     [_i, _p, _p, _p, _p, _p, _p, _p] + [_p] * 10 + [_p]),
    "dgs_debug_geometry": (_i, [_p, _i, _i, _p, _p, _p, _p, _p, _p, _p, _p]),
    "dgs_debug_binning": (_i, [_p, _p, _p, _i, _i, _i, _i, _i64, _p, _p, _p, _p]),
    "dgs_debug_image": (_i, [_p, _i, _i, _i, _p, _p, _p]),
    "dgs_debug_sort_scratch_bytes": (C.c_size_t, [_i, _i64]),
    "dgs_debug_sort": (_i, [_i, _i64, _i, _p, _p, _p, _p, _p]),
    "dgs_measure_fp32_peak": (_i, [C.POINTER(C.c_double), C.POINTER(C.c_double), _p]),
    "dgs_profile_enable": (_i, [_i]),
    "dgs_profile_num_stages": (_i, []),
    "dgs_profile_stage_name": (C.c_char_p, [_i]),
    "dgs_profile_read": (_i, [C.POINTER(C.c_double), C.POINTER(_i64), _i, _i]),
    "dgs_launch_count": (_i64, [_i]),
    "dgs_debug_workload": (_i, [_p, _p, _p, _i, _i, _i, _i, _i64, _p, _p]),
    "dgs_pose_forward": (_i, [_i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "dgs_pose_backward": (_i, [_i, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "dgs_blur_loss_forward": (_i, [_i, _i64, _p, _p, _p, _f, _p, _p, _p]),
    "dgs_blur_loss_backward": (_i, [_i, _i64, _p, _p, _p, _f, _p, _p, _p, _p]),
    "dgs_tv_loss_forward": (_i, [_i64, _i, _i, _p, _p, _p, _p]),
    "dgs_tv_loss_backward": (_i, [_i64, _i, _i, _p, _p, _p, _p]),
    "dgs_hinge_l2_forward": (_i, [_i64, _p, _p, _p, _p]),
    "dgs_hinge_l2_backward": (_i, [_i64, _p, _p, _p, _p]),
    "dgs_ssim_scratch_bytes": (C.c_size_t, [_i, _i, _i, _i]),
    "dgs_ssim_forward": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _p, _p]),
    "dgs_ssim_backward": (_i, [_i, _i, _i, _i, _p, _p, _p, _p, _i, _p, _p]),
    "dgs_activate_forward": (_i, [_i, _i, _p, _p, _p, _p, _p, _f, _i, _p, _p, _p, _p, _p]),
    "dgs_activate_backward": (_i, [_i, _i, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p]),
    "dgs_activate_forward_filter3d": (_i, [_i, _i, _p, _p, _p, _p, _p, _f, _i, _p, _p, _p, _p, _p, _p]),
    "dgs_activate_backward_filter3d": (_i, [_i, _i, _p, _p, _p, _i, _p, _p, _p, _p, _p, _p, _p, _p, _p, _f, _p,
                                            _p]),
    "dgs_filter3d_depth": (_i, [_i64, _p, _i, _p, _f, _f, _i, _i, _f, _p, _p]),
    "dgs_adam_step":(_i, [_i, _p, _p, _p, _p, C.POINTER(_i64), C.POINTER(C.c_double), C.POINTER(_i64),
                           C.c_double, C.c_double, C.c_double, C.c_double, _p]),
    "dgs_rows_gather": (_i, [_i, _p, _p, C.POINTER(_i), C.POINTER(_i), _i64, _p, _p, _p]),
    "dgs_mcmc_relocate_scratch_bytes": (C.c_size_t, [_i64]),
    "dgs_mcmc_relocate": (_i, [_i, _p, C.POINTER(_i), C.POINTER(_i), _i64, _p, _p, _p, _f, _i, _p, _p]),
    "dgs_mcmc_noise": (_i, [_i64, _p, _p, _p, _p, _f, _i, _f, _f, _f, C.c_uint64, _i64, _p]),
    "dgs_debug_mcmc_normals": (_i, [_i64, C.c_uint64, _i64, _p, _p]),
    "dgs_mark_visible": (_i, [_i, _p, _p, _p, _p, _p]),
    "dgs_knn_scratch_bytes": (C.c_size_t, [_i]),
    "dgs_knn_mean_dist2": (_i, [_i, _p, _p, _p, _p]),
}

_lib = None


class DgsError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and declare every entry point's prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DgsError(
            "libdgs_b200.so is not built (%s). Run `python -m deblurgs_b200.build` or "
            "`__graft_entry__.build()`; there is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError here = missing export: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().dgs_last_error()
        raise DgsError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else ""))


def ptr(t):
    """Device (or host) pointer of a tensor, or NULL for None / empty tensors (the reference passes
    empty CPU tensors for absent options, diff_gaussian_rasterization/__init__.py:216-226)."""
    if t is None or t.numel() == 0:
        return None
    return t.data_ptr()
