"""ctypes binding of libmvip_nerf.so (include/mvip_nerf.h).

There is no fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmvip_nerf.so")

MVIP_MLP_NUM_PARAMS = 24


class MvipPoints(ctypes.Structure):
    _fields_ = [("rays", c_void_p), ("ray_stride", c_int), ("viewdir_offset", c_int),
                ("z_vals", c_void_p), ("n_rays", c_int64), ("n_samples", c_int),
                ("pts", c_void_p), ("pts_stride", c_int64),
                ("dirs", c_void_p), ("dirs_stride", c_int64),
                ("n_points", c_int64)]


_SIGNATURES = {
    "mvip_abi_version": (c_int, []),
    "mvip_last_error": (c_char_p, []),
    "mvip_device_arch": (c_int, []),
    "mvip_rays_from_pose": (c_int, [c_void_p, c_void_p, c_int, c_int, c_float, c_float, c_float, c_int, c_int, c_int, c_int, c_int,
                                    c_void_p, c_void_p]),
    "mvip_rays_from_pose_ndc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_float, c_float, c_int, c_int, c_int, c_int,
                                        c_int, c_int, c_double, c_void_p, c_void_p]),
    "mvip_rays_pack": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_int, c_int, c_int, c_int, c_double,
                               c_double, c_void_p, c_void_p]),
    "mvip_rays_pack_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_double, c_double,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_rays_from_pose_backward_workspace_bytes": (c_size_t, []),
    "mvip_rays_from_pose_backward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_int, c_int, c_int, c_int, c_int, c_int,
                                             c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_rays_from_poses": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_double, c_float, c_float, c_int, c_int,
                                     c_double, c_void_p, c_void_p]),
    "mvip_rays_from_poses_backward_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "mvip_rays_from_poses_backward": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_double, c_int, c_int, c_double,
                                              c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_sample_coarse": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "mvip_sample_pdf": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p,
                                c_void_p, c_void_p]),
    "mvip_sample_fine": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p]),
    "mvip_composite_forward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int, c_int,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_composite_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p]),
    "mvip_composite_mse_workspace_bytes": (c_size_t, []),
    "mvip_composite_forward_mse": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_composite_backward_mse": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int, c_void_p,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_void_p]),
    "mvip_composite_backward_rays": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int64, c_int, c_int, c_int, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_void_p]),
    "mvip_normal_workspace_bytes": (c_size_t, [c_int, c_int]),
    "mvip_normal_forward": (c_int, [c_void_p, c_int, c_int, c_float, c_float, c_float, c_float, c_int, c_void_p,
                                    c_void_p, c_void_p]),
    "mvip_normal_backward": (c_int, [c_void_p, c_int, c_int, c_float, c_float, c_float, c_float, c_int, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
    "mvip_normal_forward_xyz": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "mvip_normal_backward_xyz": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_adam_step": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int,
                               c_float, c_float, c_float, c_float, c_int64, c_void_p]),
    "mvip_adam_step_dev": (c_int, [POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int,
                                   c_void_p, c_float, c_float, c_float, c_void_p, c_void_p]),
    "mvip_embed": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "mvip_mlp_packed_bytes": (c_size_t, []),
    "mvip_mlp_pack_weights": (c_int, [POINTER(c_void_p), c_void_p, c_void_p]),
    "mvip_mlp_stash_bytes": (c_size_t, [c_int64]),
    "mvip_mlp_forward": (c_int, [c_void_p, POINTER(MvipPoints), c_void_p, c_void_p, c_void_p]),
    "mvip_mlp_backward_workspace_bytes": (c_size_t, [c_int64]),
    "mvip_mlp_backward": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, POINTER(c_void_p), c_int,
                                  c_void_p]),
    "mvip_mlp_backward_phases": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, POINTER(c_void_p), c_int,
                                         c_int, c_void_p]),
    "mvip_mlp_input_grad": (c_int, [c_void_p, POINTER(MvipPoints), c_void_p, c_void_p, c_void_p, c_void_p]),
    "mvip_debug_profile": (c_int, [c_void_p]),
    "mvip_debug_trace": (c_int, [c_void_p, c_void_p]),
    "mvip_debug_wgrad_profile": (c_int, [c_void_p]),
    "mvip_debug_bwd_trace": (c_int, [c_void_p]),
    "mvip_debug_set_bwd_stagger": (c_int, [c_int]),
    "mvip_debug_bwd_lag": (c_int, [c_void_p]),
    "mvip_debug_set_bwd_throttle": (c_int, [c_int, c_int, c_int]),
    "mvip_debug_bwd_stamp_offsets": (c_int, [c_int64, c_void_p, c_void_p]),
    "mvip_selftest_umma": (c_int, [c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
}

EXPORTS = tuple(_SIGNATURES)

_lib = None


def load():
    """Loads libmvip_nerf.so once and declares every prototype of include/mvip_nerf.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError("libmvip_nerf.so not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C mvip_nerf_b200/csrc` — there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.mvip_abi_version() != 1:
        raise RuntimeError("libmvip_nerf.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().mvip_last_error()
        raise RuntimeError("%s failed (%d): %s" % (what, rc, msg.decode() if msg else "?"))
