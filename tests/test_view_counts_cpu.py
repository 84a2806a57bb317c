"""The view count at the C-ABI boundary (no GPU): every count from 1 to kMaxViews = 16 is accepted for the three shipped
flag sets in every precision (csrc/kernels.cuh: kMaxViews, csrc/model.cu validate()), 17 is refused with a message, and
the workspace a forward needs does not shrink as views are added.  The forward at these counts is checked against the
oracle in test_view_counts_gpu.py."""
import ctypes

import pytest

from openmpl_b200 import _lib, spec
from openmpl_b200.models import multiview_mpl_b200 as mb

_BASE = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=2, drop_path_rate=0.1)
ARCHS = {"hm0": dict(spec.HM0_FLAGS), "chosen": dict(spec.CHOSEN_FLAGS),
         "kptok": dict(pose_3d_emb_learnable=True, FPT_blocks_view_keypoint_tokens=True)}
PRECISIONS = ["fp32", "tf32", "bf16"]


def _create(arch, V, precision, qkv_attn_fusion=True):
    """(status, handle or None) of mpl_create for `arch` at V views."""
    desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS, **_BASE, **ARCHS[arch], num_views=V), precision,
                          qkv_attn_fusion=qkv_attn_fusion)
    h = ctypes.c_void_p()
    status = _lib.lib().mpl_create(ctypes.byref(desc), ctypes.byref(h))
    return status, (h if status == 0 else None)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("arch", list(ARCHS))
@pytest.mark.parametrize("V", [1, 16])
def test_create_accepts_one_and_sixteen_views(V, arch, precision):
    status, h = _create(arch, V, precision)
    assert status == 0, _lib.lib().mpl_last_error()
    L = _lib.lib()
    cfg = spec.make_config(**_BASE, **ARCHS[arch], num_views=V)
    assert [L.mpl_dim(h, i) for i in range(3)] == [cfg.tok_w, cfg.fpt_dim, cfg.fpt_tokens]
    assert L.mpl_workspace_bytes(h, 37) > 0 and L.mpl_packed_bytes(h) > 0
    L.mpl_destroy(h)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("arch", list(ARCHS))
def test_create_rejects_seventeen_views(arch, precision):
    status, h = _create(arch, 17, precision)
    assert h is None
    assert status == _lib.MPL_ERR_UNSUPPORTED
    msg = _lib.lib().mpl_last_error().decode()
    assert "num_views = 17" in msg and "exceeds the supported maximum of 16" in msg
    # the module creates its handle lazily and raises the library's error from there (no GPU needed to get that far)
    m = mb.MultiView_MPL(**_BASE, **ARCHS[arch], num_views=17, precision=precision).eval()
    with pytest.raises(_lib.MplError, match="exceeds the supported maximum") as err:
        m.chunk_poses()
    assert err.value.status == _lib.MPL_ERR_UNSUPPORTED


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("arch", list(ARCHS))
def test_workspace_bytes_do_not_decrease_as_views_grow(arch, precision):
    """Every per-view buffer grows with V; a workspace that shrank somewhere between 1 and 16 views would mean a buffer sized
    by a different view count than the kernels that use it.  Checked at a small batch, at the chunk size and above it.

    One buffer legitimately depends on the path rather than on V: the fused QKV + cross-view attention kernel (bf16 view
    tokens, 2 <= V <= 8, gemm_tcgen05.cu qkv_attn_supports) never materialises q|k|v, so its workspace has no q|k|v tensor
    (model.cu layout_workspace).  Monotonicity is therefore asserted with that fusion switched off, and with it on the
    workspace may only be smaller, and only at the view counts where the fused kernel runs."""
    L = _lib.lib()
    batches = (1, 37, 32768, 32768 + 1000)
    sizes = {fused: {b: [] for b in batches} for fused in (False, True)}
    for V in range(1, 17):
        for fused in (False, True):
            status, h = _create(arch, V, precision, qkv_attn_fusion=fused)
            assert status == 0, (V, _lib.lib().mpl_last_error())
            for b in batches:
                sizes[fused][b].append(L.mpl_workspace_bytes(h, b))
            L.mpl_destroy(h)
    for b, s in sizes[False].items():
        assert all(x > 0 for x in s), (b, s)
        assert s == sorted(s), (b, s)
    assert sizes[False][32768] == sizes[False][32768 + 1000]      # chunked: the workspace stops growing at one chunk
    fusable = precision == "bf16" and arch != "kptok"
    for b in batches:
        for V, (plain, fused) in enumerate(zip(sizes[False][b], sizes[True][b]), start=1):
            if fusable and 2 <= V <= 8:
                assert fused < plain, (b, V)
            else:
                assert fused == plain, (b, V)
