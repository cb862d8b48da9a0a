"""ctypes binding of libb200smpl.so (the C-ABI declared in include/b200smpl.h).

The library is hand-written CUDA for sm_100a; there is no CPU implementation behind it.  If the
shared object is missing this module raises at import-of-use time -- callers never fall back.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint8, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
# B200SMPL_LIB: an alternative build of the same library (kernel-variant experiments); never a different implementation
LIB_PATH = os.environ.get("B200SMPL_LIB") or os.path.join(HERE, "libb200smpl.so")

MODE_FP32 = 0
MODE_BF16 = 1
MODE_FP32_SIMT = 2
MODE_BF16_FAST = 3
MODES = {"fp32": MODE_FP32, "bf16": MODE_BF16, "fp32_simt": MODE_FP32_SIMT, "bf16_fast": MODE_BF16_FAST}

ERR_INVALID, ERR_CUDA, ERR_WORKSPACE = -1, -2, -3


class ModelDesc(Structure):
    _fields_ = [
        ("num_verts", c_int32), ("num_joints", c_int32), ("num_betas", c_int32),
        ("num_vertex_joints", c_int32), ("num_regressed_joints", c_int32), ("reserved0", c_int32),
        ("v_template", c_void_p), ("shapedirs", c_void_p), ("posedirs", c_void_p),
        ("J_regressor", c_void_p), ("lbs_weights", c_void_p), ("parents", c_void_p),
        ("vertex_joint_ids", c_void_p), ("joint_regressors", c_void_p),
    ]


class ModelInfo(Structure):
    _fields_ = [
        ("num_verts", c_int32), ("num_joints_out", c_int32), ("num_betas", c_int32),
        ("num_blend_rows", c_int32), ("num_blend_rows_padded", c_int32), ("feature_pitch", c_int32),
        ("num_virtual_groups", c_int32), ("device", c_int32),
    ]


class ForwardArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("mode", c_int32), ("pose_is_axis_angle", c_int32), ("slab_bodies", c_int32),
        ("betas", c_void_p), ("pose", c_void_p), ("transl", c_void_p), ("cam", c_void_p),
        ("vertices", c_void_p), ("joints", c_void_p), ("joints2d", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("saved", c_void_p), ("saved_bytes", c_size_t),
    ]


class BackwardArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("mode", c_int32), ("pose_is_axis_angle", c_int32), ("slab_bodies", c_int32),
        ("betas", c_void_p), ("pose", c_void_p), ("transl", c_void_p), ("cam", c_void_p), ("joints", c_void_p),
        ("grad_vertices", c_void_p), ("grad_joints", c_void_p), ("grad_joints2d", c_void_p),
        ("grad_betas", c_void_p), ("grad_pose", c_void_p), ("grad_transl", c_void_p), ("grad_cam", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
        ("saved", c_void_p), ("saved_bytes", c_size_t),
    ]


class FitGroup(Structure):
    _fields_ = [
        ("params", c_void_p), ("grad", c_void_p), ("grad_extra", c_void_p), ("exp_avg", c_void_p),
        ("exp_avg_sq", c_void_p), ("best_params", c_void_p), ("frozen_cols", c_void_p), ("cols", c_int32),
    ]


class MultiTaskLossArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("num_verts", c_int32), ("num_joints", c_int32), ("nmap2d", c_int32), ("nmap3d", c_int32),
        ("num_betas", c_int32), ("pose_cols", c_int32), ("reserved0", c_int32),
        ("proj_wh", c_float), ("norm_wh", c_float),
        ("verts", c_void_p), ("verts_label", c_void_p), ("joints", c_void_p), ("cam", c_void_p),
        ("map2d", c_void_p), ("label2d", c_void_p), ("vis", c_void_p), ("map3d", c_void_p), ("label3d", c_void_p),
        ("shape", c_void_p), ("shape_label", c_void_p), ("pose", c_void_p), ("pose_label", c_void_p),
        ("log_var", c_void_p), ("scratch", c_void_p),
    ]


class SilhouetteArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("num_verts", c_int32), ("num_faces", c_int32), ("img_wh", c_int32),
        ("focal_length", c_float), ("sigma", c_float),
        ("vertices", c_void_p), ("cam_t", c_void_p), ("faces", c_void_p),
        ("workspace", c_void_p), ("workspace_bytes", c_size_t),
    ]


PROXY_MAX_KEYPOINTS = 32


class ProxyArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("in_wh", c_int32), ("out_wh", c_int32), ("num_keypoints", c_int32),
        ("channels_last", c_int32), ("reserved0", c_int32), ("std", c_float),
        ("masks", c_void_p), ("keypoints", c_void_p), ("vis", c_void_p),
    ]


class ReconErrorArgs(Structure):
    _fields_ = [
        ("batch", c_int32), ("num_verts", c_int32), ("num_joints", c_int32), ("num_map", c_int32),
        ("reserved0", c_int32), ("reserved1", c_int32),
        ("pred_vertices", c_void_p), ("target_vertices", c_void_p), ("pred_joints", c_void_p),
        ("target_joints", c_void_p), ("joint_map", c_void_p),
    ]


# every symbol include/b200smpl.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "b200smpl_model_create": (c_int, [POINTER(ModelDesc), c_int, POINTER(c_void_p)]),
    "b200smpl_model_destroy": (None, [c_void_p]),
    "b200smpl_model_get_info": (c_int, [c_void_p, POINTER(ModelInfo)]),
    "b200smpl_model_debug_array": (c_int, [c_void_p, c_char_p, POINTER(c_void_p), POINTER(c_size_t)]),
    "b200smpl_saved_bytes": (c_size_t, [c_void_p, c_int, c_int]),
    "b200smpl_forward_workspace_bytes": (c_size_t, [c_void_p, c_int, c_int, c_int]),
    "b200smpl_backward_workspace_bytes": (c_size_t, [c_void_p, c_int, c_int, c_int]),
    "b200smpl_forward": (c_int, [c_void_p, POINTER(ForwardArgs), c_void_p]),
    "b200smpl_backward": (c_int, [c_void_p, POINTER(BackwardArgs), c_void_p]),
    "b200smpl_batch_rodrigues": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "b200smpl_batch_rodrigues_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200smpl_rot6d_to_rotmat": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "b200smpl_rot6d_to_rotmat_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "b200smpl_orthographic_project": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "b200smpl_orthographic_project_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                                       c_int, c_float, c_void_p]),
    "b200smpl_perspective_project": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float,
                                             c_float, c_void_p]),
    "b200smpl_perspective_project_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                      c_void_p, c_int, c_int, c_float, c_float, c_void_p]),
    "b200smpl_perspective_project_camk": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int,
                                                  c_void_p]),
    "b200smpl_perspective_project_camk_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                                           c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "b200smpl_joints2d_loss": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                       c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200smpl_fit_loss": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_float, c_float, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200smpl_fit_mark_best": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "b200smpl_fit_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_int, c_int, c_int, c_float, c_float, c_float, c_float, c_void_p]),
    "b200smpl_fit_update": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float,
                                    c_float, c_float, c_float, c_void_p]),
    "b200smpl_multitask_loss": (c_int, [POINTER(MultiTaskLossArgs), c_void_p, c_void_p]),
    "b200smpl_multitask_loss_backward": (c_int, [POINTER(MultiTaskLossArgs), c_void_p, c_void_p, c_void_p, c_void_p,
                                                 c_void_p, c_void_p, c_void_p]),
    "b200smpl_silhouette_workspace_bytes": (c_size_t, [POINTER(SilhouetteArgs)]),
    "b200smpl_silhouette_render": (c_int, [POINTER(SilhouetteArgs), c_void_p, c_void_p]),
    "b200smpl_silhouette_render_backward": (c_int, [POINTER(SilhouetteArgs), c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200smpl_silhouette_loss": (c_int, [POINTER(SilhouetteArgs), c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                         c_void_p]),
    "b200smpl_silhouette_loss_value": (c_int, [POINTER(SilhouetteArgs), c_void_p, c_float, c_void_p, c_void_p]),
    "b200smpl_proxy_representation": (c_int, [POINTER(ProxyArgs), c_void_p, c_void_p]),
    "b200smpl_reconstruction_errors": (c_int, [POINTER(ReconErrorArgs), c_void_p, c_void_p]),
    "b200smpl_debug_fwd_gemm_worklist":(c_int, [c_int, c_int, c_int, c_void_p, c_int]),
    "b200smpl_last_error": (c_char_p, []),
    "b200smpl_abi_version": (c_int, []),
    "b200smpl_launch_count": (c_int64, []),
    "b200smpl_timing_enable": (None, [c_int]),
    "b200smpl_timing_report": (c_size_t, [c_char_p, c_size_t]),
}

_lib = None


def load():
    """dlopen libb200smpl.so and type every entry point.  Raises if the library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libb200smpl.so is not built ({}). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or python soccerplayershapepose_b200/build.py). There is no CPU fallback.".format(LIB_PATH))
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.b200smpl_abi_version() != 1:
        raise RuntimeError("libb200smpl.so ABI version mismatch")
    _lib = lib
    return lib


def last_error() -> str:
    return load().b200smpl_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    """Convert a C-ABI status into the Python exceptions the reference's torch ops would raise."""
    if rc == 0:
        return
    msg = "{}: {} (code {})".format(what, last_error(), rc)
    if rc == ERR_INVALID:
        raise ValueError(msg)
    raise RuntimeError(msg)
