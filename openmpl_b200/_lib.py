"""ctypes binding of libmpl_b200.so (the C ABI declared in include/mpl_b200.h).

There is no fallback: if the shared library is missing or does not load, importing a product entry point raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MPL_B200_LIB") or os.path.join(HERE, "libmpl_b200.so")   # override: another build of the same ABI

ABI_VERSION = 9
MPL_OK = 0
MPL_ERR_INVALID_ARGUMENT = -1
MPL_ERR_CONFIG_RUNTIME = -2
MPL_ERR_CONFIG_INDEX = -3
MPL_ERR_CUDA = -4
MPL_ERR_WORKSPACE = -5
MPL_ERR_UNSUPPORTED = -6

PRECISIONS = {"fp32": 0, "tf32": 1, "bf16": 2}

# every symbol include/mpl_b200.h declares (tests check the library exports all of them)
EXPORTS = [
    "mpl_last_error", "mpl_abi_version", "mpl_create", "mpl_destroy", "mpl_num_params", "mpl_param_info", "mpl_dim",
    "mpl_packed_bytes", "mpl_pack_weights", "mpl_workspace_bytes", "mpl_chunk_poses", "mpl_set_chunk_poses",
    "mpl_forward", "mpl_last_launch_count", "mpl_mpjpe_accumulate", "mpl_build_inputs", "mpl_test_gemm",
    "mpl_set_profile", "mpl_profile_categories", "mpl_profile_category_name", "mpl_profile_collect", "mpl_synth_project",
    "mpl_pmpjpe_accumulate", "mpl_test_gemm_ln", "mpl_test_gemm_ln_slots", "mpl_test_gemm_emit_pitch", "mpl_set_graph_batch", "mpl_graph_stats",
    "mpl_test_qkv_attn", "mpl_triangulate", "mpl_triangulate_robust", "mpl_synth_detector_noise",
    "mpl_build_inputs_strided", "mpl_synth_project_strided", "mpl_synth_detector_noise_strided", "mpl_triangulate_strided",
    "mpl_triangulate_robust_strided", "mpl_synth_cameras", "mpl_triangulate_refine", "mpl_triangulate_refine_strided",
    "mpl_mpjpe_accumulate_grouped", "mpl_pmpjpe_accumulate_masked", "mpl_distort_pixels", "mpl_distort_pixels_strided",
    "mpl_undistort_pixels", "mpl_undistort_pixels_strided", "mpl_synth_calib_noise", "mpl_calibrate_rig_workspace_bytes",
    "mpl_calibrate_rig",
]

_DESC_FLAGS = [
    "qkv_bias", "add_confidence_input", "mult_confidence_emb", "concat_confidence_emb", "confidence_input_as_third",
    "pose_3d_emb_learnable", "linear_weighted_mean", "add_3D_pos_encoding_in_Spatial", "input_rays_as_token",
    "add_3D_pos_encoding_to_rays", "confidence_as_attention_uncertainty_weight", "multiple_spatial_blocks",
    "no_transformer_spt", "no_transformer_fpt", "confidence_in_FPT", "deep_head", "head_kadkhod",
    "FPT_blocks_view_keypoint_tokens",
]


class MplDesc(ctypes.Structure):
    """Mirror of `struct MplDesc` (include/mpl_b200.h)."""
    _fields_ = ([("struct_size", c_int32), ("num_joints", c_int32), ("in_chans", c_int32), ("embed_dim_ratio", c_int32),
                 ("depth", c_int32), ("num_heads", c_int32), ("num_views", c_int32), ("hidden_dim", c_int32),
                 ("mlp_ratio", c_float), ("qk_scale", c_float)]
                + [(f, c_int32) for f in _DESC_FLAGS] + [("precision", c_int32), ("ln_fusion", c_int32),
                                                         ("gemm_cta_group", c_int32), ("spt_hidden", c_int32), ("fpt_hidden", c_int32),
                                                         ("qkv_attn_fusion", c_int32),
                                                         ("chunk_streams", c_int32)])


def make_desc(kw: dict, precision: str, ln_fusion: bool = True, gemm_cta_group: int = 2, chunk_streams: int = 1,
              qkv_attn_fusion: bool = True) -> MplDesc:
    """Constructor kwargs of MultiView_MPL (multiview_mpl.py:95-117) -> MplDesc."""
    if precision not in PRECISIONS:
        raise ValueError(f"precision must be one of {sorted(PRECISIONS)}, got {precision!r}")
    d = MplDesc()
    d.struct_size = ctypes.sizeof(MplDesc)
    for f in ("num_joints", "in_chans", "embed_dim_ratio", "depth", "num_heads", "num_views", "hidden_dim"):
        setattr(d, f, int(kw[f]))
    d.mlp_ratio = float(kw["mlp_ratio"])
    d.qk_scale = float(kw["qk_scale"] or 0.0)
    for f in _DESC_FLAGS:
        setattr(d, f, int(bool(kw[f])))
    d.precision = PRECISIONS[precision]
    d.ln_fusion = int(bool(ln_fusion))
    d.gemm_cta_group = int(gemm_cta_group)
    d.chunk_streams = int(chunk_streams)
    d.qkv_attn_fusion = int(bool(qkv_attn_fusion))
    # the Mlp widths as Python's float64 int(dim * ratio) gives them (the float32 ratio in the struct can round differently)
    from .spec import make_config
    from .spec import CTOR_DEFAULTS
    cfg = make_config(**{k: v for k, v in kw.items() if k in CTOR_DEFAULTS})
    d.spt_hidden, d.fpt_hidden = int(cfg.spt_hidden), int(cfg.fpt_hidden)
    return d


class MplError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


_lib = None


def lib():
    """The loaded library; raises if it is not built (no CPU / eager fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m openmpl_b200.build` "
                               "(the MPL forward has no fallback path)")
        L = ctypes.CDLL(LIB_PATH)
        L.mpl_last_error.restype = c_char_p
        L.mpl_abi_version.restype = c_int
        L.mpl_create.argtypes = [POINTER(MplDesc), POINTER(c_void_p)]
        L.mpl_destroy.argtypes = [c_void_p]
        L.mpl_destroy.restype = None
        L.mpl_num_params.argtypes = [c_void_p]
        L.mpl_param_info.argtypes = [c_void_p, c_int, POINTER(c_char_p), POINTER(c_int64), POINTER(c_int32)]
        L.mpl_dim.argtypes = [c_void_p, c_int]
        L.mpl_dim.restype = c_int64
        L.mpl_packed_bytes.argtypes = [c_void_p]
        L.mpl_packed_bytes.restype = c_size_t
        L.mpl_pack_weights.argtypes = [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_size_t, c_void_p]
        L.mpl_workspace_bytes.argtypes = [c_void_p, c_int64]
        L.mpl_workspace_bytes.restype = c_size_t
        L.mpl_chunk_poses.argtypes = [c_void_p]
        L.mpl_chunk_poses.restype = c_int64
        L.mpl_set_chunk_poses.argtypes = [c_void_p, c_int64]
        L.mpl_forward.argtypes = [c_void_p, c_void_p, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), c_int64,
                                  c_int64, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_size_t, c_void_p]
        L.mpl_last_launch_count.argtypes = [c_void_p]
        L.mpl_last_launch_count.restype = c_int64
        L.mpl_mpjpe_accumulate.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_float, POINTER(c_float), c_void_p, c_void_p]
        L.mpl_pmpjpe_accumulate.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_float, c_int, c_int, c_void_p, c_void_p]
        L.mpl_build_inputs.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]
        L.mpl_test_gemm.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_int, c_int,
                                    c_int, c_void_p]
        L.mpl_test_gemm_ln.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p,
                                       c_int, c_void_p, c_void_p, c_float, c_int, c_int, c_int, c_void_p]
        L.mpl_test_gemm_ln_slots.argtypes = [c_int]
        L.mpl_test_gemm_emit_pitch.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p,
                                               c_int, c_int, c_int, c_void_p]
        L.mpl_test_qkv_attn.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float, c_float, c_void_p,
                                        c_int64, c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]
        L.mpl_set_graph_batch.argtypes = [c_void_p, c_int64]
        L.mpl_graph_stats.argtypes = [c_void_p, POINTER(c_int64), POINTER(c_int64)]
        L.mpl_set_profile.argtypes = [c_void_p, c_int]
        L.mpl_profile_category_name.argtypes = [c_int]
        L.mpl_profile_category_name.restype = c_char_p
        L.mpl_profile_collect.argtypes = [c_void_p, POINTER(c_double), POINTER(c_int64), c_int]
        L.mpl_synth_project.argtypes = [ctypes.c_uint64, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                        c_void_p, c_void_p]
        L.mpl_triangulate.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]
        L.mpl_triangulate_robust.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_float, c_float, c_void_p, c_void_p,
                                             c_void_p]
        L.mpl_synth_detector_noise.argtypes = [ctypes.c_uint64, c_int64, c_int64, c_int, c_int, c_void_p, c_float, c_float,
                                               c_float, c_void_p, c_void_p]
        L.mpl_build_inputs_strided.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                               c_void_p]
        L.mpl_synth_project_strided.argtypes = [ctypes.c_uint64, c_int64, c_int64, c_int, c_int, c_void_p, c_int64, c_void_p,
                                                c_int, c_void_p, c_void_p, c_void_p]
        L.mpl_triangulate_strided.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_float, c_void_p, c_void_p,
                                              c_void_p]
        L.mpl_triangulate_robust_strided.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_float, c_float,
                                                     c_void_p, c_void_p, c_void_p]
        L.mpl_synth_detector_noise_strided.argtypes = [ctypes.c_uint64, c_int64, c_int64, c_int, c_int, c_void_p, c_int64,
                                                       c_float, c_float, c_float, c_void_p, c_void_p]
        L.mpl_synth_cameras.argtypes = [ctypes.c_uint64, c_int64, c_int64, c_int, c_double, c_double, c_double, c_void_p,
                                        c_void_p, c_void_p]
        L.mpl_triangulate_refine.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_float, c_void_p, c_void_p, c_int,
                                             c_void_p, c_void_p, c_void_p]
        L.mpl_triangulate_refine_strided.argtypes = [c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_float, c_void_p,
                                                     c_void_p, c_int, c_void_p, c_void_p, c_void_p]
        L.mpl_mpjpe_accumulate_grouped.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_float,
                                                   POINTER(c_float), c_void_p, c_void_p]
        L.mpl_pmpjpe_accumulate_masked.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_float, c_int,
                                                   c_int, c_void_p, c_void_p]
        L.mpl_distort_pixels.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p]
        L.mpl_distort_pixels_strided.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int, c_int,
                                                 c_void_p]
        L.mpl_undistort_pixels.argtypes = [c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_double, c_int64, c_int, c_int,
                                           c_void_p]
        L.mpl_undistort_pixels_strided.argtypes = [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_double, c_double,
                                                   c_int64, c_int, c_int, c_void_p]
        L.mpl_synth_calib_noise.argtypes = [ctypes.c_uint64, c_int64, c_int64, c_int, c_void_p, c_int64, c_double, c_double,
                                            c_void_p, c_void_p]
        L.mpl_calibrate_rig_workspace_bytes.argtypes = [c_int64, c_int, c_int]
        L.mpl_calibrate_rig_workspace_bytes.restype = c_size_t
        L.mpl_calibrate_rig.argtypes = [c_void_p, c_void_p, c_int64, c_int, c_int, c_float, c_void_p, c_void_p, c_double,
                                        c_double, c_double, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]
        if L.mpl_abi_version() != ABI_VERSION:
            raise RuntimeError("libmpl_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(status: int):
    """Raise the Python exception class the reference would raise for this status."""
    if status == MPL_OK:
        return
    msg = lib().mpl_last_error().decode("utf-8", "replace")
    if status == MPL_ERR_CONFIG_INDEX:
        raise IndexError(msg)
    raise MplError(status, msg)
