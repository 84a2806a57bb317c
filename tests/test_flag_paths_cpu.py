"""The flag matrix of test_flag_paths_gpu.py without a GPU: every boolean constructor flag of the spec, no qkv bias, an
explicit qk_scale and an MLP ratio other than 2 each appear in at least one case, so a flag added to the spec later cannot
be left out of the matrix silently; every case is a valid configuration at production width that the library accepts in
every precision; and the matrix reaches each kernel path it exists for."""
import ctypes

import pytest

from flag_matrix import FLAG_CASES, PROD, case_kw, views_of
from gpu_util import kernel_path
from openmpl_b200 import _lib, spec

PRECISIONS = ["fp32", "tf32", "bf16"]


def test_every_flag_is_in_the_matrix():
    kws = [case_kw(n, 4) for n in FLAG_CASES]
    missing = [f for f in spec.BOOL_FLAGS if not any(kw.get(f) for kw in kws)]
    assert not missing, f"flags no case of the matrix sets: {missing}"
    assert any(kw.get("qkv_bias") is False for kw in kws)
    assert any(kw.get("qk_scale") is not None for kw in kws)
    assert any(kw.get("mlp_ratio", spec.CTOR_DEFAULTS["mlp_ratio"]) != 2.0 for kw in kws)


@pytest.mark.parametrize("name", list(FLAG_CASES))
def test_every_case_is_valid_at_production_width(name):
    for V in views_of(name):
        kw = case_kw(name, V)
        cfg = spec.make_config(**kw)
        assert cfg.error is None, cfg.error
        assert (cfg.J, cfg.d, cfg.H) == (PROD["num_joints"], PROD["embed_dim_ratio"], PROD["num_heads"])
        for precision in PRECISIONS:
            desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS, **kw), precision)
            h = ctypes.c_void_p()
            status = _lib.lib().mpl_create(ctypes.byref(desc), ctypes.byref(h))
            assert status == 0, (precision, V, _lib.lib().mpl_last_error())
            _lib.lib().mpl_destroy(h)


@pytest.mark.parametrize("path", ["spt_fused_pos_mode2", "generic_spt_ln_prep", "join_planes_view_d544",
                                  "join_planes_view_d1088", "unpermuted_interleave_planes", "permuted_planes",
                                  "fp32_tokens_no_fpt", "fused_keypoint_fpt", "confidence_weighted_fused_spt"])
def test_matrix_reaches_the_path(path):
    """Each path the matrix was built for is selected by at least one case in a tensor-core mode (gpu_util.kernel_path,
    which the GPU test checks against the profiler trace)."""
    def reached(name, V, precision):
        kw = case_kw(name, V)
        p = kernel_path(kw, precision)
        tc = precision != "fp32"
        return {
            "spt_fused_pos_mode2": tc and p["spt_fused"] and p["pos_mode2"],
            "generic_spt_ln_prep": p["ln_fused"] and p["spt"] and not p["spt_fused"],
            "join_planes_view_d544": p["join_planes"] and p["D"] == 544,
            "join_planes_view_d1088": p["join_planes"] and p["D"] == 1088,
            "unpermuted_interleave_planes": p["ln_fused"] and p["ray_layout"] == "interleave" and not p["perm"],
            "permuted_planes": p["perm"],
            "fp32_tokens_no_fpt": tc and p["spt_fused"] and not p["fpt"],
            "fused_keypoint_fpt": p["kp_fused"],
            "confidence_weighted_fused_spt": (tc and p["spt_fused"] and p["spt_apps"] > p["reps"]
                                              and precision == "tf32"),
        }[path]
    assert any(reached(n, V, pr) for n in FLAG_CASES for V in views_of(n) for pr in PRECISIONS), path
