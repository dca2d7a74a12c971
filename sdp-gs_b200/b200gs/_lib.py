"""ctypes binding of libb200gs.so (the C-ABI declared in include/b200gs.h).

There is no CPU or PyTorch fallback: if the shared library is missing or its ABI does not match
this binding, importing fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200GS_LIB: developer knob for A/B builds of the same library (tools/build_variants.sh); never a different backend
LIB_PATH = os.environ.get("B200GS_LIB") or os.path.join(_HERE, "libb200gs.so")

c_float_p = C.c_void_p  # device pointers are passed as integers


class View(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("tan_fovx", C.c_float), ("tan_fovy", C.c_float),
        ("scale_modifier", C.c_float),
        ("sh_degree", C.c_int32), ("sh_coeffs", C.c_int32),
        ("prefiltered", C.c_int32), ("debug", C.c_int32), ("extended", C.c_int32),
        ("background", C.c_void_p), ("viewmatrix", C.c_void_p), ("projmatrix", C.c_void_p), ("campos", C.c_void_p),
    ]


class Gaussians(C.Structure):
    _fields_ = [
        ("P", C.c_int32),
        ("means3D", C.c_void_p), ("shs", C.c_void_p), ("colors_precomp", C.c_void_p), ("opacities", C.c_void_p),
        ("scales", C.c_void_p), ("rotations", C.c_void_p), ("cov3D_precomp", C.c_void_p),
        ("language_feature_precomp", C.c_void_p), ("shs_language", C.c_void_p), ("confidence", C.c_void_p),
        ("live_count", C.c_void_p),
    ]


class Outputs(C.Structure):
    _fields_ = [("color", C.c_void_p), ("depth", C.c_void_p), ("alpha", C.c_void_p), ("feature", C.c_void_p),
                ("radii", C.c_void_p)]


class Workspace(C.Structure):
    _fields_ = [("geom", C.c_void_p), ("geom_bytes", C.c_size_t), ("binning", C.c_void_p),
                ("binning_bytes", C.c_size_t), ("image", C.c_void_p), ("image_bytes", C.c_size_t),
                ("persistent", C.c_int32), ("reserved_", C.c_int32)]


class GradOutputs(C.Structure):
    _fields_ = [("dL_dcolor", C.c_void_p), ("dL_ddepth", C.c_void_p), ("dL_dalpha", C.c_void_p),
                ("dL_dfeature", C.c_void_p)]


class Grads(C.Structure):
    _fields_ = [("dL_dmeans3D", C.c_void_p), ("dL_dmeans2D", C.c_void_p), ("dL_dshs", C.c_void_p),
                ("dL_dcolors", C.c_void_p), ("dL_dopacities", C.c_void_p), ("dL_dscales", C.c_void_p),
                ("dL_drotations", C.c_void_p), ("dL_dcov3D", C.c_void_p), ("dL_dfeatures", C.c_void_p),
                ("dL_dshs_language", C.c_void_p), ("scratch", C.c_void_p),
                ("scatter_bases", C.c_void_p), ("scatter_shard_rows", C.c_int64), ("scatter_rank", C.c_int32),
                ("scatter_world", C.c_int32), ("accumulate", C.c_int32), ("reserved_", C.c_int32)]


class CameraGrads(C.Structure):  # b200gs_camera_grads_t
    _fields_ = [("dL_dviewmatrix", C.c_void_p), ("dL_dprojmatrix", C.c_void_p), ("dL_dcampos", C.c_void_p),
                ("scratch", C.c_void_p)]


class HParams(C.Structure):  # include/b200gs_train.h: b200gs_hparams_t (64 bytes, lives in device memory)
    _fields_ = [("step", C.c_float), ("lr_xyz", C.c_float), ("lr_f_dc", C.c_float), ("lr_f_rest", C.c_float),
                ("lr_opacity", C.c_float), ("lr_scaling", C.c_float), ("lr_rotation", C.c_float), ("lr_feature", C.c_float),
                ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("lambda_dssim", C.c_float),
                ("depth_weight", C.c_float), ("pad", C.c_float * 3)]


_PS_GROUPS = ("xyz", "shs", "opacity", "scaling", "rotation", "feature")


class ParamState(C.Structure):  # b200gs_param_state_t
    _fields_ = ([("P", C.c_int32)]
                + [(f"{pre}{g}", C.c_void_p) for g in _PS_GROUPS for pre in ("", "m_", "v_", "g_")]
                + [("opacity_act", C.c_void_p), ("scaling_act", C.c_void_p), ("rotation_act", C.c_void_p),
                   ("g_means2D", C.c_void_p), ("radii", C.c_void_p), ("xyz_gradient_accum", C.c_void_p),
                   ("denom", C.c_void_p), ("max_radii2D", C.c_void_p)])


TRAIN_EXPORTS = ["b200gs_param_step", "b200gs_photometric_loss", "b200gs_photometric_scratch_bytes",
                 "b200gs_depth_pearson_loss", "b200gs_hparams_advance", "b200gs_loss_accum_doubles", "b200gs_knn3", "b200gs_depth_pearson_loss_pseudo", "b200gs_train_abi_sizes",
                 "b200gs_knn3_scratch_bytes", "b200gs_knn3_tree"]
COLLECTIVE_EXPORTS = ["b200gs_allreduce_sum_f32", "b200gs_allreduce_flag_words", "b200gs_gather_reduce_f32"]

EXPORTS = [
    "b200gs_version", "b200gs_last_error", "b200gs_geom_bytes", "b200gs_image_bytes", "b200gs_binning_bytes",
    "b200gs_scratch_bytes", "b200gs_workspace_init", "b200gs_forward_preprocess", "b200gs_forward_render", "b200gs_forward",
    "b200gs_forward_status", "b200gs_backward", "b200gs_mark_visible", "b200gs_geom_layout",
    "b200gs_image_layout", "b200gs_binning_layout", "b200gs_debug_sorted_keys", "b200gs_launch_count",
    "b200gs_abi_sizes", "b200gs_profile_enable", "b200gs_profile_read",
    "b200gs_backward_camera", "b200gs_camera_scratch_bytes", "b200gs_camera_grads_abi_size",
]


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `make -C sdp-gs_b200/csrc` (or __graft_entry__.build()). "
            "b200gs has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name in EXPORTS + TRAIN_EXPORTS + COLLECTIVE_EXPORTS:
        if not hasattr(lib, name):
            raise ImportError(f"{LIB_PATH} does not export {name}")
    lib.b200gs_last_error.restype = C.c_char_p
    for f in ("b200gs_geom_bytes", "b200gs_image_bytes", "b200gs_binning_bytes", "b200gs_scratch_bytes",
              "b200gs_camera_scratch_bytes"):
        getattr(lib, f).restype = C.c_size_t
    lib.b200gs_camera_scratch_bytes.argtypes = [C.c_int32]
    lib.b200gs_camera_grads_abi_size.restype = C.c_int64
    lib.b200gs_geom_bytes.argtypes = [C.c_int32]
    lib.b200gs_image_bytes.argtypes = [C.c_int32, C.c_int32]
    lib.b200gs_binning_bytes.argtypes = [C.c_int64, C.c_int32, C.c_int32]
    lib.b200gs_scratch_bytes.argtypes = [C.c_int32]
    lib.b200gs_launch_count.restype = C.c_int64
    P = C.POINTER
    lib.b200gs_workspace_init.argtypes = [P(Workspace), C.c_int32, C.c_void_p, C.c_void_p]
    lib.b200gs_forward_preprocess.argtypes = [P(View), P(Gaussians), P(Outputs), P(Workspace), C.c_void_p, P(C.c_int64)]
    lib.b200gs_forward_render.argtypes = [P(View), P(Gaussians), P(Outputs), P(Workspace), C.c_int64, C.c_void_p]
    lib.b200gs_forward.argtypes = [P(View), P(Gaussians), P(Outputs), P(Workspace), C.c_int64, C.c_void_p]
    lib.b200gs_forward_status.argtypes = [P(Workspace), C.c_void_p, P(C.c_int64), P(C.c_int32)]
    lib.b200gs_backward.argtypes = [P(View), P(Gaussians), C.c_void_p, P(Workspace), C.c_int64, P(GradOutputs), P(Grads), C.c_void_p]
    lib.b200gs_backward_camera.argtypes = [P(View), P(Gaussians), C.c_void_p, P(Workspace), C.c_int64, P(GradOutputs), P(Grads),
                                           P(CameraGrads), C.c_void_p]
    lib.b200gs_mark_visible.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.b200gs_geom_layout.argtypes = [C.c_int32, P(C.c_int64)]
    lib.b200gs_image_layout.argtypes = [C.c_int32, C.c_int32, P(C.c_int64)]
    lib.b200gs_binning_layout.argtypes = [C.c_int32, C.c_int32, C.c_int64, P(C.c_int64)]
    lib.b200gs_debug_sorted_keys.argtypes = [P(View), C.c_int32, P(Workspace), C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
    lib.b200gs_abi_sizes.argtypes = [P(C.c_int64)]
    lib.b200gs_profile_enable.argtypes = [C.c_int32]
    lib.b200gs_profile_read.argtypes = [P(C.c_double), P(C.c_int64), C.c_int32]
    lib.b200gs_param_step.argtypes = [P(ParamState), C.c_void_p, C.c_int32, C.c_void_p]
    lib.b200gs_photometric_loss.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_void_p]
    lib.b200gs_photometric_scratch_bytes.argtypes = [C.c_int32, C.c_int32]
    lib.b200gs_photometric_scratch_bytes.restype = C.c_size_t
    lib.b200gs_depth_pearson_loss.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p]
    lib.b200gs_loss_accum_doubles.restype = C.c_size_t
    lib.b200gs_depth_pearson_loss_pseudo.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                                     C.c_void_p, C.c_void_p, C.c_void_p]
    lib.b200gs_knn3.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.b200gs_knn3_scratch_bytes.argtypes = [C.c_int32]
    lib.b200gs_knn3_scratch_bytes.restype = C.c_size_t
    lib.b200gs_knn3_tree.argtypes = [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.b200gs_hparams_advance.argtypes = [C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p]
    lib.b200gs_allreduce_flag_words.argtypes = [C.c_int32]
    lib.b200gs_allreduce_flag_words.restype = C.c_size_t
    lib.b200gs_allreduce_sum_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_void_p]
    lib.b200gs_gather_reduce_f32.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    assert C.sizeof(HParams) == 64
    sizes = (C.c_int64 * 6)()
    lib.b200gs_abi_sizes(sizes)
    mine = [C.sizeof(t) for t in (View, Gaussians, Outputs, Workspace, GradOutputs, Grads)]
    if list(sizes) != mine:
        raise ImportError(f"ABI mismatch between {LIB_PATH} {list(sizes)} and this binding {mine}")
    if lib.b200gs_camera_grads_abi_size() != C.sizeof(CameraGrads):
        raise ImportError(f"ABI mismatch (camera gradients) between {LIB_PATH} {lib.b200gs_camera_grads_abi_size()} and this "
                          f"binding {C.sizeof(CameraGrads)}")
    tsizes = (C.c_int64 * 2)()
    lib.b200gs_train_abi_sizes.argtypes = [P(C.c_int64)]
    lib.b200gs_train_abi_sizes(tsizes)
    if list(tsizes) != [C.sizeof(ParamState), C.sizeof(HParams)]:
        raise ImportError(f"ABI mismatch (training structs) between {LIB_PATH} {list(tsizes)} and this binding")
    return lib


lib = _load()


class B200GSError(RuntimeError):
    pass


def check(code):
    if code != 0:
        raise B200GSError(lib.b200gs_last_error().decode("utf-8", "replace"))
