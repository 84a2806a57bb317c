"""The lifter forward at every supported view count, and on the kernel paths the goldens do not reach.

The goldens and the view sweep stop at V = 8 (oracle/cases.py), but the library accepts 1 <= V <= kMaxViews = 16 and picks
different kernels outside 2..8: the generic attention kernel for view tokens, the 14-set fused keypoint-token FPT with one
pose per CTA (V = 9..14), its 16-set / 9-warp object (V = 15, 16), the narrow or generic fp32 attention for 153..272
keypoint tokens, the head's pooling loop over 3-4 groups of four views.  Every case here is checked against the fp64 oracle
on the same seeded weights and batch, and one traced forward proves which kernels ran.  Run on the B200 with `-m gpu`."""
import functools
import gc
import json

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from conftest import load_golden
from gpu_util import DMPJPE_MM, TOL, build_module, mpjpe_mm, oracle_outputs, rel_err, run_module
from oracle.cases import CASES, make_inputs
from openmpl_b200 import spec, synth

pytestmark = pytest.mark.gpu

# fp32-grade tensor-core mode: every golden measures 5e-6 .. 2.4e-5 of scale (profiles/r2_split_mode_error_probe.log).
# 1e-4 is ~4x the worst of them and ~40x below what one lost hi.lo term of a split product costs (a bf16-grade product,
# ~2^-9 relative, i.e. 1e-3 .. 4e-3 of scale like the bf16 mode).  TOL["tf32"] = 1e-3 stays the stated contract.
TF32_GUARD = 1e-4
# bf16 at V outside the goldens: within TOL["bf16"] and within max(2 e8, 2e-3), e8 = the same architecture's error at V = 8
# (a shape the goldens pin) on the same weights, seeds and batch.  Rounding does not grow with V by 2x; a skipped or
# double-counted 17-key chunk or a view lost in the head moves the output by far more.
BF16_SIBLING_FACTOR, BF16_SIBLING_FLOOR = 2.0, 2e-3
# Weight seed of every case.  The head pools the views as sum_v w_v LN(x_v) (weighted_mean, a Conv1d over views) and
# LayerNorms the result: where sum_v w_v is near zero the pooled row nearly cancels and the head LayerNorm amplifies the
# rounding left in it, so the error measures the conditioning of the instance, not the kernels.  Seed 7 has
# sum_v w_v = +0.008 at V = 8 and +0.050 at V = 5 (bf16 errors 1.2e-2 .. 2.6e-2 there, 5-8x the neighbouring V); seed 2
# keeps |sum_v w_v| between 0.50 and 0.93 at every view count used here.  _model() refuses a seed below MIN_POOL_WEIGHT_SUM.
WEIGHT_SEED = 2
MIN_POOL_WEIGHT_SUM = 0.25


def _bf16_sibling_bound(e8):
    return max(BF16_SIBLING_FACTOR * e8, BF16_SIBLING_FLOOR)


DEPTH = 2
REPS = DEPTH + 1                       # FPT block applications per forward: the last block runs twice (model.cu FPT loop)
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
    """({kernel: (launches per forward or None, block.x or None)}, [kernels that must not run]) for one chunk at depth 2,
    d = 32, H = 8, derived from the selection conditions of the library (file:line of each next to it)."""
    flags = ARCHS[arch]
    d, H = 32, 8
    kp = bool(flags.get("FPT_blocks_view_keypoint_tokens"))
    E = J * d
    rays = bool(flags.get("input_rays_as_token"))
    D = d if kp else E * (2 if rays else 1)                                      # model.cu:823-827
    hidden = int(D * mlp_ratio)
    N = V * J if kp else V
    hd = D // H
    stacks = V if flags.get("multiple_spatial_blocks") else 1
    # model.cu:840-841 + spt_fused.cu:851: the single-kernel SPT needs J = 17, d = 32, H = 8, hidden 64 and a tensor-core mode
    spt_fused = precision != "fp32" and J == 17 and int(d * mlp_ratio) == 64
    # model.cu:843-844: the keypoint-token FPT stack as one kernel (bf16, V <= 16, same block shape as the SPT)
    kp_fused = precision == "bf16" and kp and V <= 16 and J == 17 and hidden == 64
    # model.cu:860: LayerNorm-fused bf16 mode, residual stream in two bf16 planes
    ln_fused = precision == "bf16" and not kp_fused and D % 32 == 0 and D <= 32 * 4 * 17
    must, never = {}, []
    spt_narrow = 0 if spt_fused else REPS * stacks       # generic SPT: N = J, hd = 4 -> attention_narrow_kernel
    if kp_fused:
        # spt_fused.cu:911-914: the 16-set / 9-warp object where it holds >= 25 % more of a tile than the 14-set one
        alt = 4 * ((16 // V) * V) * 14 >= 5 * ((14 // V) * V) * 16
        must["spt_fused_kernel_fast<true>"] = (1, 288 if alt else 256)
        never += ["attention_kp_h4_kernel", "attention_kernel<"]
    elif kp and precision == "bf16":
        # kernels_generic.cu:919: bf16 keypoint tokens off the fused kernel (J != 17 or hidden != 64), 8 heads of 4, N <= 272
        must["attention_kp_h4_kernel"] = (REPS, 256)
        never += ["spt_fused_kernel_fast<true>"]
    elif kp:
        # fp32 (block_f32) and tf32 (launch_attention_split -> launch_attention_any<float, float>, kernels_generic.cu:979):
        # kernels_generic.cu:937-939: whole sets in <= 96 KB of shared memory (N * 3 * 32 * 4 B) -> narrow kernel, else :955-958
        if N * 3 * D * 4 <= 96 * 1024:
            must["attention_narrow_kernel<float, float, 4>"] = (REPS + spt_narrow, 256)
            never += ["attention_kernel<"]
        else:
            must["attention_kernel<float, float>"] = (REPS, 128)
            if spt_narrow:
                must["attention_narrow_kernel<float, float, 4>"] = (spt_narrow, 256)
            else:
                never += ["attention_narrow_kernel"]
        if precision == "tf32":
            must["to_split_kernel"] = (None, None)                               # kernels_generic.cu:980
    else:
        # model.cu:864 + gemm_tcgen05.cu:1250-1253: fused QKV + attention for 136- or 68-wide heads and 2 <= V <= 8
        qkv_attn = ln_fused and (D == H * 136 or (D == H * 68 and H % 2 == 0)) and 2 <= V <= 8
        # kernels_generic.cu:903-913 (and :977 for tf32): the K4 view kernel for 2 <= N <= 8 wide heads
        views = 2 <= V <= 8 and hd >= 16 and hd % 4 == 0 and D // 4 <= 288 and D // 4 >= H * N
        if qkv_attn:
            must["qkv_attn_kernel"] = (REPS, None)
        elif views:
            must["attention_views_kernel"] = (REPS, None)
        else:
            # kernels_generic.cu:955-958: one warp per (set, head, query), wide-head branch (hd > 16)
            t = "__nv_bfloat16, __nv_bfloat16" if precision == "bf16" else "float, float"
            must[f"attention_kernel<{t}>"] = (REPS, 128)
            never += ["qkv_attn_kernel", "attention_views_kernel"]
            if precision == "tf32":
                must["to_split_kernel"] = (None, None)                           # kernels_generic.cu:972-980
    if spt_fused:
        if not kp:
            never += ["attention_narrow_kernel"]         # the SPT is the only narrow-head attention of view tokens
    else:
        never += ["spt_fused_kernel_fast<false>", "spt_fused_kernel_precise"]
    # model.cu:684-685 / 632-633: ln_prep converts the fp32 tokens into the planes unless the fused SPT wrote them
    if ln_fused:
        if spt_fused:
            never += ["ln_prep_kernel"]
        else:
            must["ln_prep_kernel"] = (1, None)
    # head: model.cu:704-705 (ray-layout rows are read as 32-channel segments at stride 64 unless the planes are channel-
    # permuted, model.cu:871-872), model.cu:632 + 711-714 (planes are read directly), io_kernels.cu:447 (instantiation)
    ray_layout1 = rays and bool(flags.get("add_3D_pos_encoding_to_rays"))
    perm = ln_fused and ray_layout1 and spt_fused and D == 2 * E
    stride = 64 if (ray_layout1 and not perm) else 32
    nk = f"9, {stride}, 17" if E == 544 else ("9, 0, 0" if E > 320 else "5, 0, 0")
    must[f"head_block_kernel<{nk}, {'true' if ln_fused else 'false'}>"] = (1, 256)
    return must, never


def _normalise(name):
    return name.replace("(bool)1", "true").replace("(bool)0", "false")


def _traced_forward(m, batch, tmp_path):
    """Output of one forward and [(kernel name, block.x)] of every kernel it launched (graph_batch=0: no graph replay)."""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run_module(m, batch)
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    kernels = [(_normalise(e["name"]), (e.get("args", {}).get("block") or [None])[0])
               for e in events if e.get("cat") == "kernel"]
    assert kernels, "the trace holds no kernel events"
    return out, kernels


def _check_kernels(kernels, must, never, label):
    seen = []
    for key, (count, block) in must.items():
        hits = [(n, b) for n, b in kernels if key in n]
        assert hits, f"{label}: {key} did not run; kernels: {sorted({n for n, _ in kernels})}"
        if count is not None:
            assert len(hits) == count, f"{label}: {key} ran {len(hits)} times, expected {count}"
        if block is not None:
            assert {b for _, b in hits} == {block}, f"{label}: {key} blocks {sorted({b for _, b in hits})}, expected {block}"
        seen.append(f"{key}x{len(hits)}" + (f"/b{block}" if block else ""))
    for key in never:
        hits = sorted({n for n, _ in kernels if key in n})
        assert not hits, f"{label}: {key} must not run here, ran: {hits}"
    return " ".join(seen)


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
    outs, kernels = _traced_forward(m, batch, tmp_path)
    out = outs[0]
    assert out.shape == (B_SMALL, 17, 3) and np.isfinite(out).all()
    e = rel_err(out, ref)
    dmm = _dmpjpe(out, ref, batch["target"])
    bound = _bound(precision)
    sib = ""
    if precision == "bf16":
        bound = min(bound, _bf16_sibling_bound(e8(arch)))
        sib = f" e8 {e8(arch):.3e}"
    label = f"{arch} V={V} {precision}"
    ran = _check_kernels(kernels, *_expected(arch, precision, V), label)
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
        bound = min(bound, _bf16_sibling_bound(e8(arch)))
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
    out, kernels = _traced_forward(m, batch, tmp_path)
    e = rel_err(out[0], ref)
    dmm = _dmpjpe(out[0], ref, batch["target"])
    bound = TOL["bf16"]
    if V == 16:
        bound = min(bound, _bf16_sibling_bound(_plain_error("kptok", 4, "bf16", J, mlp_ratio)))
    label = f"kptok J={J} mlp_ratio={mlp_ratio} V={V} bf16"
    ran = _check_kernels(kernels, *_expected("kptok", "bf16", V, J, mlp_ratio), label)
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
    out, kernels = _traced_forward(m, batch, tmp_path)
    assert out[0].shape == (B_SMALL, 13, 3)
    e = rel_err(out[0], ref)
    dmm = _dmpjpe(out[0], ref, batch["target"])
    label = f"hm0 J=13 V={V} {precision}"
    ran = _check_kernels(kernels, *_expected("hm0", precision, V, 13), label)
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
