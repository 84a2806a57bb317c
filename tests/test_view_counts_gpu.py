"""The lifter forward at every supported view count, and on the kernel paths the goldens do not reach.

The goldens and the view sweep stop at V = 8 (oracle/cases.py), but the library accepts 1 <= V <= kMaxViews = 16 and picks
different kernels outside 2..8: the generic attention kernel for view tokens, the 14-set fused keypoint-token FPT with one
pose per CTA (V = 9..14), its 16-set / 9-warp object (V = 15, 16), the narrow or generic fp32 attention for 153..272
keypoint tokens, the head's pooling loop over 3-4 groups of four views.  Every case here is checked against the fp64 oracle
on the same seeded weights and batch, and one traced forward proves which kernels ran.  Run on the B200 with `-m gpu`."""
import functools
import gc

import numpy as np
import pytest
import torch

from conftest import load_golden
from gpu_util import (DMPJPE_MM, MIN_POOL_WEIGHT_SUM, TF32_GUARD, TOL, WEIGHT_SEED, bf16_sibling_bound, build_module,
                      check_kernels, expected_kernels, mpjpe_mm, oracle_outputs, rel_err, run_module, traced_forward)
from oracle.cases import CASES, make_inputs
from openmpl_b200 import spec, synth

pytestmark = pytest.mark.gpu

DEPTH = 2
B_SMALL = 37                           # ragged CTA tiles everywhere (14-set SPT tiles, 16-pose head groups, 128-row GEMMs)
VIEWS = [1, 9, 11, 14, 15, 16]
PRECISIONS = ["fp32", "tf32", "bf16"]
CHUNK = 32768                          # default forward chunk (model.cu MplModel::chunk)
_BASE = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=DEPTH, drop_rate=0.0, attn_drop_rate=0.0,
             drop_path_rate=0.1)
ARCHS = {"hm0": dict(spec.HM0_FLAGS),                     # view tokens, D = 1088 ([x_j | ray_j] per joint), per-view SPT stacks
         "chosen": dict(spec.CHOSEN_FLAGS),               # view tokens, D = 544, 68-wide heads
         "kptok": dict(pose_3d_emb_learnable=True, FPT_blocks_view_keypoint_tokens=True)}   # V * J tokens of width 32


def _model(arch, V, J=17, mlp_ratio=2.0):
    kw = dict(_BASE, **ARCHS[arch], num_views=V, num_joints=J, mlp_ratio=mlp_ratio)
    cfg = spec.make_config(**kw)
    weights = synth.named_weights(spec.param_spec(cfg), seed=WEIGHT_SEED)
    wsum = float(np.sum(weights["weighted_mean.weight"]))
    assert abs(wsum) >= MIN_POOL_WEIGHT_SUM, f"ill-conditioned view pooling at V = {V}: sum of weights {wsum:.3f}"
    return kw, cfg, weights


def _batch(V, B, J=17, seed=11):
    batch = synth.make_batch(B, synth.make_rig(V), seed=seed)
    if J != synth.NUM_JOINTS:                    # same slicing as oracle.cases.make_inputs
        batch = {k: np.ascontiguousarray(v[:, :, :J] if k in ("poses", "rays") else v[:, :J] if k == "target" else v)
                 for k, v in batch.items()}
    return batch


@functools.lru_cache(maxsize=None)
def _case(arch, V, J=17, mlp_ratio=2.0):
    """(kw, cfg, weights, batch, fp64 oracle output) of the B_SMALL-pose case; the same seeds for every V and precision."""
    kw, cfg, weights = _model(arch, V, J, mlp_ratio)
    batch = _batch(V, B_SMALL, J)
    return kw, cfg, weights, batch, oracle_outputs(cfg, weights, batch)[0]


@functools.lru_cache(maxsize=None)
def _plain_error(arch, V, precision, J=17, mlp_ratio=2.0):
    kw, cfg, weights, batch, ref = _case(arch, V, J, mlp_ratio)
    return rel_err(run_module(build_module(kw, weights, precision, graph_batch=0), batch)[0], ref)


@pytest.fixture(scope="module")
def e8():
    """bf16 error at V = 8 of each architecture, measured in this session on the weights / seeds / batch of the sweep."""
    def get(arch):
        e = _plain_error(arch, 8, "bf16")
        # V = 8 is a shape the goldens pin: its error must be inside the bf16 contract, or the sibling rule measures nothing
        assert e <= TOL["bf16"], f"{arch} bf16 at V = 8: {e:.3e} of scale"
        return e
    return get


def _bound(precision):
    return TF32_GUARD if precision == "tf32" else TOL[precision]


# ---- which kernels a forward must launch ------------------------------------------------------------------------------
def _expected(arch, precision, V, J=17, mlp_ratio=2.0):
    """gpu_util.expected_kernels for one case of this file (selection conditions and their file:line there)."""
    return expected_kernels(dict(_BASE, **ARCHS[arch], num_views=V, num_joints=J, mlp_ratio=mlp_ratio), precision)


def _dmpjpe(out, ref, target):
    t = target.astype(np.float64)
    return abs(mpjpe_mm(out, t) - mpjpe_mm(ref, t))


# ---- 1. the view-count matrix -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("V", VIEWS)
@pytest.mark.parametrize("arch", list(ARCHS))
def test_forward_at_view_count_matches_oracle_on_its_kernel_path(arch, V, precision, e8, tmp_path):
    kw, cfg, weights, batch, ref = _case(arch, V)
    m = build_module(kw, weights, precision, graph_batch=0)
    outs, kernels = traced_forward(m, batch, tmp_path)
    out = outs[0]
    assert out.shape == (B_SMALL, 17, 3) and np.isfinite(out).all()
    e = rel_err(out, ref)
    dmm = _dmpjpe(out, ref, batch["target"])
    bound = _bound(precision)
    sib = ""
    if precision == "bf16":
        bound = min(bound, bf16_sibling_bound(e8(arch)))
        sib = f" e8 {e8(arch):.3e}"
    label = f"{arch} V={V} {precision}"
    ran = check_kernels(kernels, *_expected(arch, precision, V), label)
    print(f"[view-counts] {label}: err {e:.3e} of scale (bound {bound:.1e}{sib}), dMPJPE {dmm:.4f} mm | {ran}")
    assert e <= bound, f"{label}: {e:.3e} of scale > {bound:.1e}"
    assert dmm <= DMPJPE_MM[precision], f"{label}: dMPJPE {dmm:.4f} mm"


# ---- 1b. size-independent properties at V = 16 ------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["tf32", "bf16"])
@pytest.mark.parametrize("arch", ["hm0", "kptok"])
def test_sixteen_views_two_chunk_batch_is_pose_independent(arch, precision, e8):
    """32 768 + 1 000 poses at V = 16: two forward chunks, the second ragged.  A full chunk of view tokens is 524 288 FPT rows
    and the tf32 q|k|v of hm0 is 1.71e9 fp32 values (under 2^31 = 2.15e9 elements, but 6.8 GB): the generic attention
    kernel's row offsets and every pointer into that tensor address past 2 GB, so a byte offset computed in 32 bits would
    break; an int32 element index would not overflow here.  Sampled poses
    (first and last 8, both sides of the chunk boundary, random ones) match the oracle; the same poses alone give the same
    bits; a 256-pose batch on the CUDA-graph path gives the bits of the plain path."""
    V = 16
    kw, cfg, weights = _model(arch, V)
    B = CHUNK + 1000
    batch = synth.make_batch(B, synth.make_rig(V), seed=42)
    m = build_module(kw, weights, precision)
    assert m.chunk_poses() == CHUNK
    out = run_module(m, batch, packed=True)[0]
    assert out.shape == (B, 17, 3) and np.isfinite(out).all()
    rng = np.random.default_rng(0)
    idx = np.unique(np.concatenate([np.arange(8), np.arange(B - 8, B), np.arange(CHUNK - 8, CHUNK + 8),
                                    rng.choice(B, 40, replace=False)]))
    sub = {k: np.ascontiguousarray(v[idx]) for k, v in batch.items()}
    ref = oracle_outputs(cfg, weights, sub)[0]
    e = rel_err(out[idx], ref)
    dmm = _dmpjpe(out[idx], ref, sub["target"])
    bound = _bound(precision)
    if precision == "bf16":
        bound = min(bound, bf16_sibling_bound(e8(arch)))
    print(f"[view-counts] {arch} V=16 {precision} B={B} ({len(idx)} sampled poses): err {e:.3e} of scale (bound {bound:.1e}), "
          f"dMPJPE {dmm:.4f} mm")
    assert e <= bound, f"{arch} [{precision}] B={B}: {e:.3e}"
    assert dmm <= DMPJPE_MM[precision]
    alone = run_module(m, sub, packed=True)[0]
    np.testing.assert_array_equal(alone, out[idx])
    del m
    gc.collect()
    torch.cuda.empty_cache()
    small = {k: v[:256] for k, v in batch.items()}
    plain = build_module(kw, weights, precision, graph_batch=0)
    graph = build_module(kw, weights, precision, graph_batch=512)
    a = run_module(plain, small)[0]
    b = run_module(graph, small)[0]
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(a, out[:256])
    assert graph.graph_stats() == (1, 0) and plain.graph_stats() == (0, 0)


# ---- 2. branches the view count alone does not reach ------------------------------------------------------------------
@pytest.mark.parametrize("V", [4, 16])
@pytest.mark.parametrize("J,mlp_ratio", [(13, 2.0), (17, 3.0)], ids=["j13", "hidden96"])
def test_bf16_keypoint_tokens_off_the_fused_kernel(J, mlp_ratio, V, tmp_path):
    """bf16 keypoint tokens the fused FPT kernel cannot take (J != 17, or hidden 96) run attention_kp_h4_kernel: N = 13 V is
    not a multiple of its 17-key chunk; J = 17 at V = 16 is N = 272, the launcher's limit.  V = 16 must also stay within
    max(2 e4, 2e-3) of the V = 4 error of the same configuration."""
    kw, cfg, weights, batch, ref = _case("kptok", V, J, mlp_ratio)
    m = build_module(kw, weights, "bf16", graph_batch=0)
    out, kernels = traced_forward(m, batch, tmp_path)
    e = rel_err(out[0], ref)
    dmm = _dmpjpe(out[0], ref, batch["target"])
    bound = TOL["bf16"]
    if V == 16:
        bound = min(bound, bf16_sibling_bound(_plain_error("kptok", 4, "bf16", J, mlp_ratio)))
    label = f"kptok J={J} mlp_ratio={mlp_ratio} V={V} bf16"
    ran = check_kernels(kernels, *_expected("kptok", "bf16", V, J, mlp_ratio), label)
    print(f"[view-counts] {label}: err {e:.3e} of scale (bound {bound:.1e}), dMPJPE {dmm:.4f} mm | {ran}")
    assert e <= bound, f"{label}: {e:.3e}"
    assert dmm <= DMPJPE_MM["bf16"]


@pytest.mark.parametrize("V", [4, 16])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_hm0_flags_with_thirteen_joints(precision, V, tmp_path):
    """J = 13 (E = 416, D = 832): the head is head_block_kernel<9, 0, 0, PL> (bf16 reads unpermuted planes: the permutation
    needs the fused SPT, model.cu:871), and the SPT leaves the fused kernel for the generic path plus ln_prep."""
    kw, cfg, weights, batch, ref = _case("hm0", V, 13)
    m = build_module(kw, weights, precision, graph_batch=0)
    out, kernels = traced_forward(m, batch, tmp_path)
    assert out[0].shape == (B_SMALL, 13, 3)
    e = rel_err(out[0], ref)
    dmm = _dmpjpe(out[0], ref, batch["target"])
    label = f"hm0 J=13 V={V} {precision}"
    ran = check_kernels(kernels, *_expected("hm0", precision, V, 13), label)
    print(f"[view-counts] {label}: err {e:.3e} of scale (bound {_bound(precision):.1e}), dMPJPE {dmm:.4f} mm | {ran}")
    assert e <= _bound(precision), f"{label}: {e:.3e}"
    assert dmm <= DMPJPE_MM[precision]


# ---- 3. the fp32-grade guard over the goldens -------------------------------------------------------------------------
TC_CASES = [n for n in CASES if not CASES[n]["kw"].get("no_transformer_fpt")]


@pytest.mark.parametrize("name", TC_CASES)
def test_tf32_goldens_within_fp32_grade_guard(name):
    """tf32 mode against the reference goldens at 1e-4 of scale (TF32_GUARD): catches a lost hi.lo term in a split GEMM or
    in the PRECISE SPT, which the 1e-3 contract would let through."""
    case = CASES[name]
    g = load_golden(name)
    cfg, weights, batch = make_inputs(case)
    out = run_module(build_module(case["kw"], weights, "tf32"), batch)[0]
    e = rel_err(out, g["out64_0"])
    print(f"[tf32-guard] {name}: err {e:.3e} of scale (bound {TF32_GUARD:.0e})")
    assert e <= TF32_GUARD, f"{name} [tf32]: {e:.3e} of scale"
