"""The lifter forward under every constructor flag at production width, on the kernel path each flag takes.

The flag goldens (oracle/cases.py, `flag_*`) are built at d = 16, H = 4, where no tensor-core mode runs the kernels that
serve the flags in production: the single-kernel SPT needs J = 17, d = 32, H = 8, hidden 64 (spt_fused.cu:851) and the
LayerNorm-fused bf16 FPT needs a width that is a multiple of 32 (model.cu:857).  Here every flag case of the goldens
(tests/flag_matrix.py) runs at d = 32, H = 8, J = 17, depth 2, B = 37 (ragged CTA tiles everywhere), V = 4 (and V = 5
where the FPT runs on D = 544 / 1088 view tokens), in fp32, tf32 and bf16, against the fp64 oracle on the same seeded
weights and batch.  One traced forward per case proves which kernels ran.  Run on the B200 with `-m gpu`."""
import functools

import numpy as np
import pytest
import torch

from flag_matrix import FLAG_CASES, SIBLINGS, case_kw, sibling_of, views_of
from gpu_util import (DMPJPE_MM, MIN_POOL_WEIGHT_SUM, TF32_GUARD, TOL, WEIGHT_SEED, bf16_sibling_bound, build_module,
                      check_kernels, expected_kernels, kernel_path, mpjpe_mm, oracle_outputs, pool_weight_sum, rel_err,
                      run_module, traced_forward)
from openmpl_b200 import spec, synth

pytestmark = pytest.mark.gpu

B_SMALL = 37
PRECISIONS = ["fp32", "tf32", "bf16"]
MATRIX = [(n, V) for n in FLAG_CASES for V in views_of(n)]


def _model(kw):
    cfg = spec.make_config(**kw)
    assert cfg.error is None, cfg.error
    weights = synth.named_weights(spec.param_spec(cfg), seed=WEIGHT_SEED)
    wsum = pool_weight_sum(weights)          # None for linear_weighted_mean: no per-view pooling weight to cancel
    assert wsum is None or abs(wsum) >= MIN_POOL_WEIGHT_SUM, f"ill-conditioned view pooling: sum of weights {wsum:.3f}"
    return cfg, weights


@functools.lru_cache(maxsize=None)
def _case(name, V):
    """(kw, cfg, weights, batch, fp64 oracle outputs) of the B_SMALL-pose case; the same seeds for every precision."""
    kw = case_kw(name, V)
    cfg, weights = _model(kw)
    batch = synth.make_batch(B_SMALL, synth.make_rig(V), seed=11)
    return kw, cfg, weights, batch, oracle_outputs(cfg, weights, batch)


@functools.lru_cache(maxsize=None)
def _sibling_error(arch, V):
    """bf16 error of the golden-pinned architecture of one FPT kind on this file's seeds, batch and V."""
    kw = dict(case_kw("plain", V), **SIBLINGS[arch])
    cfg, weights = _model(kw)
    batch = synth.make_batch(B_SMALL, synth.make_rig(V), seed=11)
    e = rel_err(run_module(build_module(kw, weights, "bf16", graph_batch=0), batch)[0], oracle_outputs(cfg, weights, batch)[0])
    # a shape the goldens pin: its error must be inside the bf16 contract, or the sibling rule measures nothing
    assert e <= TOL["bf16"], f"{arch} bf16 at V = {V}: {e:.3e} of scale"
    return e


def _bound(name, V, precision):
    """(bound, note): TF32_GUARD in tf32; in bf16 TOL["bf16"] and max(2 e_sibling, 2e-3)."""
    if precision == "tf32":
        return TF32_GUARD, ""
    if precision == "fp32":
        return TOL["fp32"], ""
    arch = sibling_of(name, V)
    es = _sibling_error(arch, V)
    return min(TOL["bf16"], bf16_sibling_bound(es)), f" {arch} {es:.3e}"


def _flag_expected(kw, precision):
    """expected_kernels plus the flag-dependent front and back of the forward (file:line of each condition)."""
    must, never = expected_kernels(kw, precision)
    p = kernel_path(kw, precision)
    if p["spt_fused"]:
        # model.cu:638-645: one launch for the whole SPT stack of every view; PRECISE in tf32, fast<false> in bf16
        must["spt_fused_kernel_precise" if precision == "tf32" else "spt_fused_kernel_fast<false>"] = (1, None)
        never += ["spt_fused_kernel_fast<false>" if precision == "tf32" else "spt_fused_kernel_precise"]
        never += ["token_build"]                          # model.cu:622 + 668: its epilogue writes the FPT tokens
    else:
        must["token_build"] = (1, 256)                    # model.cu:668 (token_build_vec_kernel or token_build_kernel)
        if not p["kp"]:
            if p["spt"]:
                # model.cu:650-662: generic SPT, N = J = 17, hd = 4 -> attention_narrow_kernel once per block application
                # (the confidence-weighted pass included) and stack; the FPT of view tokens has no narrow heads
                must["attention_narrow_kernel<float, float, 4>"] = (p["spt_apps"] * p["stacks"], 256)
            else:
                never += ["attention_narrow_kernel"]
    # model.cu:621 + 635: a stand-alone embed kernel unless the fused SPT computes the embedding in its prologue, which it
    # does for every spatial position mode but Linear(normalize(ray)) (spatial_pos_mode 2, model.cu:577)
    if p["fuse_embed"]:
        never += ["embed_"]
    else:
        must["embed_"] = (1, 256)                         # embed_vec_kernel or embed_kernel
    # model.cu:704-709: non-K5 heads behind the bf16 planes refill the fp32 tokens once
    if p["join_planes"]:
        must["join_planes_kernel"] = (1, None)
    else:
        never += ["join_planes_kernel"]
    return must, never


def _dmpjpe(out, ref, target):
    t = target.astype(np.float64)
    return abs(mpjpe_mm(out, t) - mpjpe_mm(ref, t))


# ---- 1. the flag matrix -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name,V", MATRIX, ids=[f"{n}-V{V}" for n, V in MATRIX])
def test_flag_case_matches_oracle_on_its_kernel_path(name, V, precision, tmp_path):
    kw, cfg, weights, batch, refs = _case(name, V)
    m = build_module(kw, weights, precision, graph_batch=0)
    outs, kernels = traced_forward(m, batch, tmp_path)
    assert len(outs) == len(refs) == (3 if kw.get("head_kadkhod") else 1)   # head_kadkhod: (x, [x1, x2])
    for o in outs:
        assert o.shape == (B_SMALL, 17, 3) and np.isfinite(o).all()
    errs = [rel_err(o, r) for o, r in zip(outs, refs)]
    e = max(errs)
    dmm = _dmpjpe(outs[0], refs[0], batch["target"])
    bound, note = _bound(name, V, precision)
    label = f"{name} V={V} {precision}"
    p = kernel_path(kw, precision)
    must, never = _flag_expected(kw, precision)
    # the tensor-core paths this matrix exists for: the fused view attention where the FPT runs on view tokens, the fused
    # keypoint-token FPT in bf16
    if precision != "fp32" and p["fpt"] and not p["kp"]:
        assert ("qkv_attn_kernel" if precision == "bf16" else "attention_views_kernel") in must, label
    if precision == "bf16" and p["fpt"] and p["kp"]:
        assert "spt_fused_kernel_fast<true>" in must, label
    ran = check_kernels(kernels, must, never, label)
    outs_note = "" if len(errs) == 1 else " (x1 {:.3e}, x2 {:.3e})".format(*errs[1:])
    print(f"[flag-paths] {label}: err {e:.3e} of scale{outs_note} (bound {bound:.1e}{note}), dMPJPE {dmm:.4f} mm | {ran}")
    assert e <= bound, f"{label}: {e:.3e} of scale > {bound:.1e}"
    assert dmm <= DMPJPE_MM[precision], f"{label}: dMPJPE {dmm:.4f} mm"


# ---- 1b. the generic head behind the planes, against the K5 head on the same FPT output -------------------------------
# Against the oracle, the bf16 error of the whole forward (~2e-3 of scale) hides anything the size of one bf16 rounding:
# join_planes_kernel returning the hi plane alone raises the error of the non-K5 heads by 1.1 .. 1.7x (to at most 3.3e-3
# of scale, B200), inside max(2 e_sibling, 2e-3).  This test compares the generic head with the K5 head on identical FPT output
# instead: linear_weighted_mean with weight kron(w, I_E) and bias b is the Conv1d view mean sum_v w_v x_v + b, so the
# "linmean" flag set (no rays: no channel permutation, the same FPT kernels as the default head) and its default-head
# twin compute the same function and share every kernel up to the head.  The K5 head reads hi + lo from the planes, the
# generic chain reads them through join_planes_kernel; both heads are fp32-grade, so the outputs must agree to 1e-4.
HEAD_TWIN_BOUND = 1e-4


@pytest.mark.parametrize("V", [4, 5])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_generic_head_equals_k5_head_on_the_same_tokens(precision, V, tmp_path):
    kw_lin = case_kw("linmean", V)
    kw_k5 = dict(kw_lin, linear_weighted_mean=False)
    cfg, w_k5 = _model(kw_k5)
    w_lin = {k: v for k, v in w_k5.items() if not k.startswith("weighted_mean.")}
    w_lin["weighted_mean.weight"] = np.kron(w_k5["weighted_mean.weight"].reshape(1, V), np.eye(cfg.E)).astype(np.float32)
    w_lin["weighted_mean.bias"] = np.full(cfg.E, w_k5["weighted_mean.bias"][0], np.float32)
    batch = synth.make_batch(B_SMALL, synth.make_rig(V), seed=11)
    k5 = run_module(build_module(kw_k5, w_k5, precision, graph_batch=0), batch)[0]
    out, kernels = traced_forward(build_module(kw_lin, w_lin, precision, graph_batch=0), batch, tmp_path)
    label = f"linmean twin V={V} {precision}"
    ran = check_kernels(kernels, *_flag_expected(kw_lin, precision), label)
    d = rel_err(out[0], k5.astype(np.float64))
    print(f"[flag-paths] {label}: generic head vs K5 head {d:.3e} of scale (bound {HEAD_TWIN_BOUND:.0e}) | {ran}")
    assert d <= HEAD_TWIN_BOUND, f"{label}: {d:.3e} of scale"


# ---- 2. size-independent properties on the newly reached paths --------------------------------------------------------
@pytest.mark.parametrize("name,precision", [("hm0flags_deephead", "bf16"), ("hm0flags_kadkhod", "bf16"),
                                            ("confattn_multi", "tf32")])
def test_large_batch_is_pose_independent(name, precision):
    """3000 packed poses at V = 4 (many GEMM / SPT / head tiles, ragged tails): poses sampled from both ends and at random
    match the oracle, and the same poses run alone give the same bits, every output of head_kadkhod included."""
    V, B = 4, 3000
    kw = case_kw(name, V)
    cfg, weights = _model(kw)
    batch = synth.make_batch(B, synth.make_rig(V), seed=42)
    m = build_module(kw, weights, precision)
    outs = run_module(m, batch, packed=True)
    rng = np.random.default_rng(0)
    idx = np.unique(np.concatenate([np.arange(8), np.arange(B - 8, B), rng.choice(B, 48, replace=False)]))
    sub = {k: np.ascontiguousarray(v[idx]) for k, v in batch.items()}
    refs = oracle_outputs(cfg, weights, sub)
    bound = TF32_GUARD if precision == "tf32" else TOL[precision]
    errs = [rel_err(o[idx], r) for o, r in zip(outs, refs)]
    dmm = _dmpjpe(outs[0][idx], refs[0], sub["target"])
    print(f"[flag-paths] {name} V={V} {precision} B={B} ({len(idx)} sampled poses): err "
          f"{' / '.join(f'{e:.3e}' for e in errs)} of scale (bound {bound:.1e}), dMPJPE {dmm:.4f} mm")
    assert all(np.isfinite(o).all() for o in outs)
    assert max(errs) <= bound, f"{name} [{precision}] B={B}: {errs}"
    assert dmm <= DMPJPE_MM[precision]
    alone = run_module(m, sub, packed=True)
    assert len(alone) == len(outs)
    for a, o in zip(alone, outs):
        np.testing.assert_array_equal(a, o[idx])


def _kadkhod():
    kw = case_kw("hm0flags_kadkhod", 4)
    return kw, *_model(kw)


def test_kadkhod_chunked_and_pipelined_equal_one_call():
    """head_kadkhod writes three outputs per chunk (x1, x2 at the chunk's pose offset, model.cu mpl_forward chunk loop).
    1000 poses in 256-pose chunks (1000 = 3 * 256 + 232), from device memory and from pinned host memory (the module's
    pipelined chunk loop), must give every output bitwise as one device-resident call does."""
    kw, cfg, weights = _kadkhod()
    batch = synth.make_batch(1000, synth.make_rig(4), seed=12)
    m = build_module(kw, weights, "bf16", graph_batch=0)
    ref = run_module(m, batch, packed=True)
    assert len(ref) == 3 and all(np.isfinite(r).all() for r in ref)
    m.set_chunk_poses(256)
    chunked = run_module(m, batch, packed=True)
    args = [torch.from_numpy(batch[k]).pin_memory() for k in ("poses", "rays", "centers")]
    with torch.no_grad():
        out, aux = m(args[0], rays=args[1], centers=args[2])
    torch.cuda.synchronize()
    piped = [out.cpu().numpy()] + [a.cpu().numpy() for a in aux]
    for i in range(3):
        np.testing.assert_array_equal(chunked[i], ref[i], err_msg=f"output {i}, device-resident chunks")
        np.testing.assert_array_equal(piped[i], ref[i], err_msg=f"output {i}, pipelined host chunks")


def test_kadkhod_cuda_graph_equals_plain_path():
    """256 poses on the CUDA-graph path (graph_batch = 512) give all three outputs bitwise as the kernel-by-kernel path."""
    kw, cfg, weights = _kadkhod()
    batch = synth.make_batch(256, synth.make_rig(4), seed=13)
    plain = build_module(kw, weights, "bf16", graph_batch=0)
    graph = build_module(kw, weights, "bf16", graph_batch=512)
    a = run_module(plain, batch)
    b = run_module(graph, batch)
    assert len(a) == len(b) == 3
    for i in range(3):
        np.testing.assert_array_equal(a[i], b[i], err_msg=f"output {i}")
    assert graph.graph_stats() == (1, 0) and plain.graph_stats() == (0, 0)
