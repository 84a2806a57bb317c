"""CPU-side checks of the C-ABI boundary and the host module: the library loads and exports every symbol the header
declares, its parameter table is the reference's state_dict, invalid flag combinations fail like the reference, and the
product path refuses to run without a GPU (no fallback).  No compute calls here."""
import ctypes
import itertools
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden
from oracle import ref_loader
from oracle.cases import CASES, GRID_BASE, GRID_FLAGS
from openmpl_b200 import _lib, spec
from openmpl_b200.models import multiview_mpl_b200 as mb


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "mpl_b200.h")).read()
    declared = set(re.findall(r"\b(mpl_[a-z0-9_]+)\s*\(", header))
    declared.discard("mpl_stream_t")
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), name
    assert _lib.lib().mpl_abi_version() == _lib.ABI_VERSION


def _lib_param_table(kw, precision="fp32"):
    L = _lib.lib()
    full = dict(spec.CTOR_DEFAULTS)
    full.update(kw)
    desc = _lib.make_desc(full, precision)
    h = ctypes.c_void_p()
    status = L.mpl_create(ctypes.byref(desc), ctypes.byref(h))
    if status != 0:
        return status, None
    name, numel, is_int = ctypes.c_char_p(), ctypes.c_int64(), ctypes.c_int32()
    table = []
    for i in range(L.mpl_num_params(h)):
        assert L.mpl_param_info(h, i, ctypes.byref(name), ctypes.byref(numel), ctypes.byref(is_int)) == 0
        table.append((name.value.decode(), numel.value, bool(is_int.value)))
    dims = [L.mpl_dim(h, i) for i in range(7)]
    L.mpl_destroy(h)
    return 0, (table, dims)


@pytest.mark.parametrize("name", list(CASES))
def test_param_table_matches_state_dict_spec(name):
    kw = CASES[name]["kw"]
    cfg = spec.make_config(**kw)
    status, (table, dims) = _lib_param_table(kw)
    assert status == 0
    want = [(n, int(np.prod(s)) if len(s) else 1, k == "count") for n, (s, k, _) in spec.param_spec(cfg).items()]
    assert table == want
    assert dims[:6] == [cfg.tok_w, cfg.fpt_dim, cfg.fpt_tokens, cfg.E, cfg.spt_hidden, cfg.fpt_hidden]


def test_create_rejects_what_the_reference_rejects():
    """mpl_create fails on exactly the flag combinations whose first forward raises in the reference (Q6 grid)."""
    ok = load_golden("validity_grid")["ok"]
    for idx, bits in enumerate(itertools.product((False, True), repeat=len(GRID_FLAGS))):
        status, _ = _lib_param_table(dict(GRID_BASE, **dict(zip(GRID_FLAGS, bits))))
        assert (status == 0) == bool(ok[idx]), (bits, status)
        if status != 0:
            assert status in (_lib.MPL_ERR_CONFIG_RUNTIME, _lib.MPL_ERR_CONFIG_INDEX)
            assert _lib.lib().mpl_last_error()


def test_bad_struct_size_and_precision_are_rejected():
    L = _lib.lib()
    desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS), "fp32")
    h = ctypes.c_void_p()
    desc.struct_size = 12
    assert L.mpl_create(ctypes.byref(desc), ctypes.byref(h)) == _lib.MPL_ERR_INVALID_ARGUMENT
    desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS), "fp32")
    desc.precision = 9
    assert L.mpl_create(ctypes.byref(desc), ctypes.byref(h)) == _lib.MPL_ERR_INVALID_ARGUMENT
    # fields kept for the struct layout: each accepts 0 and the one schedule that exists (CTA pairs, the caller's stream)
    for field, good, bad in (("gemm_cta_group", (0, 2), (1, 3)), ("chunk_streams", (0, 1), (2, -1))):
        for value in good + bad:
            desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS), "fp32")
            setattr(desc, field, value)
            status = L.mpl_create(ctypes.byref(desc), ctypes.byref(h))
            if value in good:
                assert status == 0, (field, value)
                L.mpl_destroy(h)
            else:
                assert status == _lib.MPL_ERR_INVALID_ARGUMENT, (field, value)
                assert field in L.mpl_last_error().decode()
    # tensor-core modes refuse widths the tcgen05 kernel cannot tile instead of silently falling back
    kw = dict(spec.CTOR_DEFAULTS, num_joints=13, embed_dim_ratio=8, num_heads=2, num_views=3)     # D = 104
    desc = _lib.make_desc(kw, "bf16")
    assert L.mpl_create(ctypes.byref(desc), ctypes.byref(h)) == _lib.MPL_ERR_UNSUPPORTED


def test_workspace_and_packed_sizes_are_monotone():
    L = _lib.lib()
    desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS, depth=2, num_views=4, **spec.HM0_FLAGS), "bf16")
    h = ctypes.c_void_p()
    assert L.mpl_create(ctypes.byref(desc), ctypes.byref(h)) == 0
    sizes = [L.mpl_workspace_bytes(h, b) for b in (1, 7, 100, 5000, 32768, 65536, 10 ** 7)]
    assert sizes == sorted(sizes) and sizes[-1] == sizes[-2] == sizes[-3]      # chunked: stops growing at the chunk size
    assert L.mpl_packed_bytes(h) > 4 * sum(int(np.prod(s)) for s, k, _ in spec.param_spec(spec.make_config(
        depth=2, num_views=4, **spec.HM0_FLAGS)).values() if k != "count")
    assert L.mpl_set_chunk_poses(h, 0) != 0 and L.mpl_set_chunk_poses(h, 1000) == 0
    assert L.mpl_chunk_poses(h) == 1000
    L.mpl_destroy(h)


def test_module_state_dict_names_and_ctor_signature():
    import inspect
    sig = inspect.signature(mb.MultiView_MPL.__init__)
    names = [p for p, q in sig.parameters.items() if p != "self" and q.kind != q.KEYWORD_ONLY]   # keyword-only = implementation switches
    assert names == list(spec.CTOR_DEFAULTS)
    for k, v in spec.CTOR_DEFAULTS.items():
        assert sig.parameters[k].default == v, k
    kw = CASES["flag_kadkhod"]["kw"]
    m = mb.MultiView_MPL(**kw)
    sd = m.state_dict()
    want = spec.param_spec(spec.make_config(**kw))
    assert list(sd.keys()) == list(want.keys())
    for k, (shape, kind, _) in want.items():
        assert tuple(sd[k].shape) == tuple(shape), k


@pytest.mark.skipif(not ref_loader.available(), reason="/root/reference not mounted")
@pytest.mark.parametrize("name", ["hm0_v4_d12", "flag_kadkhod", "flag_deephead", "flag_addmultconf_multi", "flag_linmean",
                                  "flag_confattn", "flag_kptok", "flag_nospt_nofpt", "flag_noqkvbias_scale"])
def test_state_dict_round_trips_with_the_reference_module(name):
    """Keys, shapes and dtypes equal the unmodified reference module's; its state_dict loads strictly."""
    ref = ref_loader.load_model_module()
    kw = CASES[name]["kw"]
    torch.manual_seed(0)
    r = ref.MultiView_MPL(**kw)
    m = mb.MultiView_MPL(**kw)
    rsd, msd = r.state_dict(), m.state_dict()
    assert list(rsd.keys()) == list(msd.keys())
    for k in rsd:
        assert rsd[k].shape == msd[k].shape and rsd[k].dtype == msd[k].dtype, k
    m.load_state_dict(rsd, strict=True)
    r.load_state_dict(m.state_dict(), strict=True)


def test_default_init_follows_pytorch_defaults():
    torch.manual_seed(1)
    m = mb.MultiView_MPL(depth=1, num_views=2, pose_3d_emb_learnable=True)
    sd = m.state_dict()
    assert float(sd["Spatial_pos_embed"].abs().max()) == 0 and float(sd["pos_3d_embed"].abs().max()) == 0   # Q5
    w = sd["blocks.0.attn.qkv.weight"]
    bound = 1.0 / np.sqrt(w.shape[1])
    assert float(w.abs().max()) <= bound and float(w.abs().max()) > 0.9 * bound
    assert torch.all(sd["blocks.0.norm1.weight"] == 1) and torch.all(sd["blocks.0.norm1.bias"] == 0)
    assert all(not p.requires_grad for p in m.parameters())


def test_g_wrapper_num_views_rule_and_factory():
    """MultiView_MPL_G's num_views rule (multiview_mpl.py:534-546) on a config object shaped like the reference's."""
    from types import SimpleNamespace as NS

    def cfg(test_ds="multiview_h36m_mpl", train_views=None, helper=False, helper_views=None, all_tr=False, all_te=False, n_all=7):
        net = NS(NUM_JOINTS=17, DIM=16, TRANSFORMER_DEPTH=1, TRANSFORMER_HEADS=4, TRANSFORMER_DROP_RATE=0.0,
                 TRANSFORMER_ATTN_DROP_RATE=0.0, TRANSFORMER_DROP_PATH_RATE=0.1, TRANSFORMER_ADD_CONFIDENCE_INPUT=False,
                 TRANSFORMER_MULT_CONFIDENCE_EMB=False, TRANSFORMER_CONCAT_CONFIDENCE_EMB=False,
                 TRANSFORMER_CONFIDENCE_INPUT_AS_THIRD=True, POSE_3D_EMB_LEARNABLE=True, TRANSFORMER_LINEAR_WEIGHTED_MEAN=False,
                 TRANSFORMER_ADD_3D_POS_ENCODING_IN_SPATIAL=False, TRANSFORMER_INPUT_RAYS_AS_TOKEN=True,
                 TRANSFORMER_ADD_3D_POS_ENCODING_TO_RAYS=True, TRANSFORMER_CONF_ATTENTION_UNCERTAINTY_WEIGHT=False,
                 TRANSFORMER_MULTIPLE_SPATIAL_BLOCKS=True, TRANSFORMER_NO_SPT=False, TRANSFORMER_NO_FPT=False,
                 TRANSFORMER_CONFIDENCE_IN_FPT=False, TRANSFORMER_OUTPUT_HEAD_DEEP=False, TRANSFORMER_OUTPUT_HEAD_KADKHOD=False,
                 TRANSFORMER_OUTPUT_HEAD_HIDDEN_DIM=64, TRANSFORMER_FPT_BLOCKS_VIEW_KEYPOINT_TOKENS=False,
                 INIT_WEIGHTS_FROM="scratch", INIT_WEIGHTS=True, PRETRAINED="")
        ds = NS(TEST_DATASET=test_ds, TRAIN_VIEWS=train_views, USE_HELPER_CAMERAS=helper, TRAIN_VIEWS_HELPER=helper_views,
                TRAIN_ON_ALL_CAMERAS=all_tr, TEST_ON_ALL_CAMERAS=all_te, N_VIEWS_TRAIN_TEST_ALL=n_all)
        return NS(NETWORK=net, DATASET=ds)

    assert mb.get_multiview_mpl_net(cfg(), is_train=False).features.num_views == 4
    assert mb.get_multiview_mpl_net(cfg("multiview_cmu_panoptic_mpl"), is_train=True).features.num_views == 5
    assert mb.MultiView_MPL_G(cfg("multiview_amass_cmu_panoptic_mpl")).features.num_views == 5
    assert mb.MultiView_MPL_G(cfg(train_views=[1, 3])).features.num_views == 2
    assert mb.MultiView_MPL_G(cfg(train_views=[1, 3], helper=True, helper_views=[2, 4, 5])).features.num_views == 5
    assert mb.MultiView_MPL_G(cfg(all_tr=True, all_te=True)).features.num_views == 7
    g = mb.MultiView_MPL_G(cfg())
    assert all(k.startswith("features.") for k in g.state_dict())


@pytest.mark.skipif(not ref_loader.available(), reason="/root/reference not mounted")
def test_g_wrapper_accepts_the_reference_yaml_configs():
    """The shipped YAMLs, parsed by the reference's own config module, build the same architecture in both wrappers."""
    C = ref_loader.load_config_module()
    ref = ref_loader.load_model_module()
    import glob
    yamls = sorted(glob.glob(os.path.join(ref_loader.REF_ROOT, "MPL/configs/*/mpl_amass/*.yaml")))
    assert yamls
    import contextlib, io
    for y in yamls[:2]:
        C.update_config(y)
        with contextlib.redirect_stdout(io.StringIO()):
            r = ref.MultiView_MPL_G(C.config)
        m = mb.get_multiview_mpl_net(C.config, is_train=False)
        assert list(r.state_dict().keys()) == list(m.state_dict().keys()), y
        assert all(a.shape == b.shape for a, b in zip(r.state_dict().values(), m.state_dict().values()))


def _small_cfg():
    from types import SimpleNamespace as NS
    net = NS(NUM_JOINTS=17, DIM=16, TRANSFORMER_DEPTH=2, TRANSFORMER_HEADS=4, TRANSFORMER_DROP_RATE=0.0,
             TRANSFORMER_ATTN_DROP_RATE=0.0, TRANSFORMER_DROP_PATH_RATE=0.1, TRANSFORMER_ADD_CONFIDENCE_INPUT=False,
             TRANSFORMER_MULT_CONFIDENCE_EMB=False, TRANSFORMER_CONCAT_CONFIDENCE_EMB=False,
             TRANSFORMER_CONFIDENCE_INPUT_AS_THIRD=True, POSE_3D_EMB_LEARNABLE=True, TRANSFORMER_LINEAR_WEIGHTED_MEAN=False,
             TRANSFORMER_ADD_3D_POS_ENCODING_IN_SPATIAL=False, TRANSFORMER_INPUT_RAYS_AS_TOKEN=True,
             TRANSFORMER_ADD_3D_POS_ENCODING_TO_RAYS=True, TRANSFORMER_CONF_ATTENTION_UNCERTAINTY_WEIGHT=False,
             TRANSFORMER_MULTIPLE_SPATIAL_BLOCKS=True, TRANSFORMER_NO_SPT=False, TRANSFORMER_NO_FPT=False,
             TRANSFORMER_CONFIDENCE_IN_FPT=False, TRANSFORMER_OUTPUT_HEAD_DEEP=False, TRANSFORMER_OUTPUT_HEAD_KADKHOD=False,
             TRANSFORMER_OUTPUT_HEAD_HIDDEN_DIM=64, TRANSFORMER_FPT_BLOCKS_VIEW_KEYPOINT_TOKENS=False,
             INIT_WEIGHTS_FROM="scratch", INIT_WEIGHTS=True, PRETRAINED="")
    ds = NS(TEST_DATASET="multiview_h36m_mpl", TRAIN_VIEWS=None, USE_HELPER_CAMERAS=False, TRAIN_VIEWS_HELPER=None,
            TRAIN_ON_ALL_CAMERAS=False, TEST_ON_ALL_CAMERAS=False, N_VIEWS_TRAIN_TEST_ALL=7)
    return NS(NETWORK=net, DATASET=ds)


@pytest.mark.skipif(not ref_loader.available(), reason="/root/reference not mounted")
def test_reference_checkpoint_files_load_like_valid_mpl(tmp_path):
    """The two files the reference's `save_checkpoint` writes (utils.py:148-153) -- `checkpoint.pth.tar` = a dict with
    'state_dict' of the DataParallel-unwrapped MultiView_MPL_G, `model_best.pth.tar` = the bare state_dict -- load into
    the drop-in the way `valid_mpl.py:164-175` and `load_checkpoint` (utils.py:121-126) load them."""
    import contextlib, io
    ref = ref_loader.load_model_module()
    cfg = _small_cfg()
    torch.manual_seed(3)
    with contextlib.redirect_stdout(io.StringIO()):
        r = ref.MultiView_MPL_G(cfg)
    for p_ in r.parameters():                                   # "trained" values: nothing left at its init value
        p_.data.add_(0.01 * torch.randn_like(p_))
    states = {"epoch": 7, "state_dict": r.state_dict(), "perf": 1.0, "optimizer": {}}
    torch.save(states, tmp_path / "checkpoint.pth.tar")
    torch.save(states["state_dict"], tmp_path / "model_best.pth.tar")
    # valid_mpl.py:171-175: model.load_state_dict(torch.load(model_state_file), strict=False)
    m = mb.get_multiview_mpl_net(cfg, is_train=False)
    res = m.load_state_dict(torch.load(tmp_path / "model_best.pth.tar"), strict=False)
    assert not res.missing_keys and not res.unexpected_keys
    for (k, a), (k2, b) in zip(r.state_dict().items(), m.state_dict().items()):
        assert k == k2 and torch.equal(a, b), k
    # utils.py:121-126: model.module.load_state_dict(checkpoint['state_dict']) on the DataParallel wrapper
    m2 = torch.nn.DataParallel(mb.get_multiview_mpl_net(cfg, is_train=False), device_ids=None)
    ck = torch.load(tmp_path / "checkpoint.pth.tar")
    m2.module.load_state_dict(ck["state_dict"])
    assert ck["epoch"] == 7 and all(torch.equal(a, b) for a, b in zip(r.state_dict().values(), m2.module.state_dict().values()))
    # and back: a checkpoint written from the drop-in loads strictly into the reference module
    torch.save(m.state_dict(), tmp_path / "final_state.pth.tar")
    r.load_state_dict(torch.load(tmp_path / "final_state.pth.tar"), strict=True)


def test_forward_refuses_training_mode_invalid_flags_and_missing_gpu():
    m = mb.MultiView_MPL(depth=1, num_views=2, embed_dim_ratio=8, num_heads=2)
    x = [torch.zeros(2, 17, 3)] * 2
    c = [torch.zeros(2, 1, 3)] * 2
    with pytest.raises(RuntimeError, match="inference-only"):
        m(x, rays=x, centers=c)
    m.eval()
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            m(x, rays=x, centers=c)
    bad = mb.MultiView_MPL(depth=1, num_views=2, embed_dim_ratio=8, num_heads=2, no_transformer_spt=True,
                           multiple_spatial_blocks=True).eval()
    with pytest.raises(IndexError):
        bad(x, rays=x, centers=c)
    bad = mb.MultiView_MPL(depth=1, num_views=2, embed_dim_ratio=8, num_heads=2, add_3D_pos_encoding_to_rays=True).eval()
    with pytest.raises(RuntimeError):
        bad(x, rays=x, centers=c)
    with pytest.raises(TypeError):
        mb.MultiView_MPL(not_a_kwarg=1)


def test_product_path_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under openmpl_b200/ may import or reference it."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "openmpl_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), os.path.join(dirpath, f)
                assert "mpl_oracle" not in text, os.path.join(dirpath, f)


def test_missing_library_fails_loudly_without_fallback(tmp_path):
    """No CPU / eager fallback: with the shared library absent (MPL_B200_LIB pointing nowhere) the first use raises."""
    import subprocess
    import sys
    code = ("import os, sys; sys.path.insert(0, %r); "
            "from openmpl_b200.models import multiview_mpl_b200 as mb; "
            "m = mb.MultiView_MPL(depth=1, num_views=2); "
            "from openmpl_b200 import _lib; _lib.lib()") % ROOT
    env = dict(os.environ, MPL_B200_LIB=str(tmp_path / "nowhere" / "libmpl_b200.so"))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
    assert "is missing" in r.stderr and "no fallback" in r.stderr


def test_mlp_hidden_width_follows_float64_like_the_reference():
    """int(dim * mlp_ratio) in float64 (multiview_mpl.py:25-26,78): ratio 0.7 with width 10 gives 7; the float32 ratio of the
    struct alone would give 6 and the parameter tables would disagree (ADVICE r1)."""
    L = _lib.lib()
    kw = dict(spec.CTOR_DEFAULTS, num_joints=5, embed_dim_ratio=10, num_heads=2, depth=1, num_views=2, mlp_ratio=0.7)
    desc = _lib.make_desc(kw, "fp32")
    h = ctypes.c_void_p()
    assert L.mpl_create(ctypes.byref(desc), ctypes.byref(h)) == 0, L.mpl_last_error()
    assert L.mpl_dim(h, 4) == int(10 * 0.7) == 7 and L.mpl_dim(h, 5) == int(50 * 0.7)
    L.mpl_destroy(h)
    m = mb.MultiView_MPL(**{k: v for k, v in kw.items()})
    assert m.state_dict()["Spatial_blocks.0.mlp.fc1.weight"].shape == (7, 10)


def test_depth_zero_skips_the_head_divisibility_checks():
    """With depth 0 the reference builds no blocks, so a width that is not divisible by the head count is legal."""
    cfg = spec.make_config(num_joints=5, embed_dim_ratio=10, num_heads=4, depth=0, num_views=2)
    assert cfg.error is None
    L = _lib.lib()
    desc = _lib.make_desc(dict(spec.CTOR_DEFAULTS, num_joints=5, embed_dim_ratio=10, num_heads=4, depth=0, num_views=2), "fp32")
    h = ctypes.c_void_p()
    assert L.mpl_create(ctypes.byref(desc), ctypes.byref(h)) == 0, L.mpl_last_error()
    L.mpl_destroy(h)


def test_pipelined_staging_pieces_cover_the_batch_once_and_in_order():
    """Host inputs larger than a forward chunk are copied piece by piece under the kernels of the previous piece
    (multiview_mpl_b200._forward_pipelined): a short first piece, then whole chunks."""
    from openmpl_b200.models.multiview_mpl_b200 import pipeline_pieces
    assert pipeline_pieces(65536, 32768, 4096) == [(0, 4096), (4096, 36864), (36864, 65536)]
    assert pipeline_pieces(1000, 256, 100) == [(0, 100), (100, 356), (356, 612), (612, 868), (868, 1000)]
    assert pipeline_pieces(1000, 256, 10 ** 9) == [(0, 256), (256, 512), (512, 768), (768, 1000)]      # never more than a chunk
    assert pipeline_pieces(300, 256, 0) == [(0, 1), (1, 257), (257, 300)]
    for B, chunk, first in [(1, 1, 1), (7, 3, 2), (32769, 32768, 4096), (4096, 32768, 4096), (5, 100, 100)]:
        pieces = pipeline_pieces(B, chunk, first)
        assert pieces[0][0] == 0 and pieces[-1][1] == B
        assert all(a[1] == b[0] for a, b in zip(pieces, pieces[1:]))
        assert all(0 < b1 - b0 <= chunk for b0, b1 in pieces)
