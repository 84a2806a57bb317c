"""Helpers shared by the -m gpu parity tests (the oracle is only ever the checker)."""
import json

import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import mpl_oracle
from openmpl_b200 import spec
from openmpl_b200.models import multiview_mpl_b200 as mb

# Stated tolerances (per-coordinate max abs error / output scale), BASELINE.json north_star:
#   fp32  : CUDA-core fp32 arithmetic (measured ~1e-6)
#   tf32  : the fp32-grade TENSOR-CORE mode that carries the north-star claim "<= 1e-3 of scale, dMPJPE <= 0.1 mm for the
#           fp32/TF32 path": tcgen05 on split bf16 hi/lo operands (three MMAs per product), fp32 everything else
#   bf16  : bf16 tensor-core operands, fp32 accumulate / LayerNorm statistics / softmax / residual.  Measured 1.0e-3 ..
#           4.1e-3 on the shipped architectures, 1.0e-2 on the worst parity case -> stated bound 1.2e-2, 0.5 mm
TOL = {"fp32": 2e-5, "tf32": 1e-3, "bf16": 1.2e-2}
DMPJPE_MM = {"fp32": 0.1, "tf32": 0.1, "bf16": 0.5}     # |MPJPE(new) - MPJPE(reference)| in mm (targets in metres)
# fp32-grade tensor-core mode: every golden measures 5e-6 .. 2.4e-5 of scale (profiles/r2_split_mode_error_probe.log).
# 1e-4 is ~4x the worst of them and ~40x below what one lost hi.lo term of a split product costs (a bf16-grade product,
# ~2^-9 relative, i.e. 1e-3 .. 4e-3 of scale like the bf16 mode).  TOL["tf32"] = 1e-3 stays the stated contract.
TF32_GUARD = 1e-4
# bf16 off the goldens: within TOL["bf16"] and within max(2 e, 2e-3), e = the error of a golden-pinned sibling (the same
# architecture at V = 8, or the shipped architecture of the same FPT kind) on the same weights, seeds and batch.  Rounding
# does not grow by 2x between siblings; a skipped or double-counted term moves the output by far more.
BF16_SIBLING_FACTOR, BF16_SIBLING_FLOOR = 2.0, 2e-3
# Weight seed of the synthetic-batch cases.  The head pools the views as sum_v w_v LN(x_v) (weighted_mean, a Conv1d over
# views) and LayerNorms the result: where sum_v w_v is near zero the pooled row nearly cancels and the head LayerNorm
# amplifies the rounding left in it, so the error measures the conditioning of the instance, not the kernels.  Seed 7 has
# sum_v w_v = +0.008 at V = 8 and +0.050 at V = 5 (bf16 errors 1.2e-2 .. 2.6e-2 there, 5-8x the neighbouring V); seed 2
# keeps |sum_v w_v| between 0.50 and 0.93 at every view count used.  pool_weight_sum() lets a test refuse a seed below
# MIN_POOL_WEIGHT_SUM.
WEIGHT_SEED = 2
MIN_POOL_WEIGHT_SUM = 0.25


def bf16_sibling_bound(e_sibling):
    return max(BF16_SIBLING_FACTOR * e_sibling, BF16_SIBLING_FLOOR)


def pool_weight_sum(weights):
    """sum_v w_v of the weighted_mean Conv1d, or None for linear_weighted_mean (a full Linear, no per-view weight)."""
    w = weights.get("weighted_mean.weight")
    return None if w is None or w.ndim != 3 else float(np.sum(w))


def build_module(kw, weights, precision, device="cuda", **impl):
    m = mb.MultiView_MPL(**kw, precision=precision, **impl)
    m.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in weights.items()}, strict=True)
    return m.to(device).eval()


def run_module(m, batch, packed=False, device="cuda"):
    V = batch["poses"].shape[1]
    if packed:
        args = [torch.from_numpy(batch[k]).to(device) for k in ("poses", "rays", "centers")]
    else:
        args = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])).to(device) for v in range(V)]
                for k in ("poses", "rays", "centers")]
    with torch.no_grad():
        out = m(args[0], rays=args[1], centers=args[2])
    torch.cuda.synchronize()
    if isinstance(out, tuple):
        return [out[0].cpu().numpy()] + [o.cpu().numpy() for o in out[1]]
    return [out.cpu().numpy()]


def oracle_outputs(cfg, weights, batch):
    out = mpl_oracle.forward(weights, cfg, batch["poses"], batch["rays"], batch["centers"])
    return [out[0]] + list(out[1]) if isinstance(out, tuple) else [out]


def rel_err(a, ref):
    scale = max(float(np.abs(ref).max()), 1e-6)
    return float(np.abs(a.astype(np.float64) - ref).max()) / scale


def mpjpe_mm(pred, target):
    return float(np.sqrt(((pred.astype(np.float64) - target) ** 2).sum(-1)).mean()) * 1000.0


# ---- which kernels a forward launches ---------------------------------------------------------------------------------
def kernel_path(kw, precision):
    """The kernel-selection decisions of mpl_create for constructor kwargs `kw` (file:line of each condition beside it)."""
    c = spec.make_config(**kw)
    J, V, d, H, depth, E = c.J, c.V, c.d, c.H, c.depth, c.E
    D, N = c.fpt_dim, c.fpt_tokens
    p = dict(J=J, V=V, d=d, H=H, depth=depth, E=E, D=D, N=N, hd=D // H, hidden=c.fpt_hidden, reps=depth + 1,
             kp=bool(kw.get("FPT_blocks_view_keypoint_tokens")), ray_layout=c.ray_layout)
    p["spt"] = not kw.get("no_transformer_spt") and depth > 0
    p["fpt"] = not kw.get("no_transformer_fpt") and depth > 0
    p["stacks"] = V if kw.get("multiple_spatial_blocks") else 1
    # model.cu:666-667 (spt_fused.cu:366 in the fused SPT): one more SPT block application per layer for the
    # confidence-weighted pass
    p["spt_apps"] = p["reps"] + (depth if kw.get("confidence_as_attention_uncertainty_weight") else 0)
    # model.cu:840-841 + spt_fused.cu:851: the single-kernel SPT needs J = 17, d = 32, H = 8, hidden 64 and a tensor-core mode
    p["spt_fused"] = precision != "fp32" and p["spt"] and J == 17 and d == 32 and H == 8 and c.spt_hidden == 64
    # model.cu:843-844: the keypoint-token FPT stack as one kernel (bf16, V <= 16, same block shape as the SPT)
    p["kp_fused"] = (precision == "bf16" and p["kp"] and p["fpt"] and V <= 16 and J == 17 and D == 32 and H == 8
                     and p["hidden"] == 64)
    # model.cu:846 + 860: LayerNorm-fused bf16 mode, residual stream in two bf16 planes (model.cu:632: `planes`)
    p["ln_fused"] = precision == "bf16" and p["fpt"] and not p["kp_fused"] and D % 32 == 0 and D <= 32 * 4 * 17
    # model.cu:864 + gemm_tcgen05.cu:1250-1253: fused QKV + attention for 136- or 68-wide heads and 2 <= V <= 8
    p["qkv_attn"] = p["ln_fused"] and (D == H * 136 or (D == H * 68 and H % 2 == 0)) and 2 <= N <= 8
    # model.cu:628: the SPT kernel computes the embedding unless the 3D position is Linear(normalize(ray)) (model.cu:584)
    p["pos_mode2"] = bool(kw.get("add_3D_pos_encoding_in_Spatial")) and not kw.get("pose_3d_emb_learnable")
    p["fuse_embed"] = p["spt_fused"] and not p["pos_mode2"]
    # model.cu:707: the K5 head (head_fused / head_block_kernel) serves the default head only
    p["fused_head"] = not (kw.get("linear_weighted_mean") or kw.get("deep_head") or kw.get("head_kadkhod"))
    # model.cu:870-872: channel-permuted planes need the interleaved ray layout, the fused SPT and the K5 head
    p["perm"] = (p["ln_fused"] and c.ray_layout == "interleave" and p["spt_fused"] and D == 2 * E and p["fused_head"])
    # model.cu:711-716: every head but the K5 one reading the planes refills the fp32 tokens from them
    p["join_planes"] = p["ln_fused"] and not p["fused_head"]
    return p


def expected_kernels(kw, precision):
    """({kernel: (launches per forward or None, block.x or None)}, [kernels that must not run]) for one chunk of the
    forward configured by `kw`, derived from the selection conditions of the library (file:line of each next to it)."""
    p = kernel_path(kw, precision)
    V, N, D, H, hd, REPS, kp = p["V"], p["N"], p["D"], p["H"], p["hd"], p["reps"], p["kp"]
    must, never = {}, []
    # generic SPT: N = J, hd = 4 -> attention_narrow_kernel (also with the confidence scaling, kernels_generic.cu:937-947)
    spt_narrow = p["spt_apps"] * p["stacks"] if p["spt"] and not p["spt_fused"] else 0
    if p["kp_fused"]:
        # spt_fused.cu:911-914: the 16-set / 9-warp object where it holds >= 25 % more of a tile than the 14-set one
        alt = 4 * ((16 // V) * V) * 14 >= 5 * ((14 // V) * V) * 16
        must["spt_fused_kernel_fast<true>"] = (1, 288 if alt else 256)
        never += ["attention_kp_h4_kernel", "attention_kernel<"]
    elif kp and p["fpt"] and precision == "bf16":
        # kernels_generic.cu:919: bf16 keypoint tokens off the fused kernel (J != 17 or hidden != 64), 8 heads of 4, N <= 272
        must["attention_kp_h4_kernel"] = (REPS, 256)
        never += ["spt_fused_kernel_fast<true>"]
    elif kp and p["fpt"]:
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
    elif p["fpt"]:
        # kernels_generic.cu:903-913 (and :977 for tf32): the K4 view kernel for 2 <= N <= 8 wide heads
        views = 2 <= V <= 8 and hd >= 16 and hd % 4 == 0 and D // 4 <= 288 and D // 4 >= H * N
        if p["qkv_attn"]:
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
    else:
        # no FPT (model.cu:679): the only attention left is the SPT's
        never += ["qkv_attn_kernel", "attention_views_kernel", "attention_kernel<", "attention_kp_h4_kernel",
                  "spt_fused_kernel_fast<true>"]
        if spt_narrow:
            must["attention_narrow_kernel<float, float, 4>"] = (spt_narrow, 256)
        else:
            never += ["attention_narrow_kernel"]
    if p["spt_fused"]:
        if not kp:
            never += ["attention_narrow_kernel"]         # the SPT is the only narrow-head attention of view tokens
    else:
        never += ["spt_fused_kernel_fast<false>", "spt_fused_kernel_precise"]
    # model.cu:684-685 / 632-633: ln_prep converts the fp32 tokens into the planes unless the fused SPT wrote them
    if p["ln_fused"]:
        if p["spt_fused"]:
            never += ["ln_prep_kernel"]
        else:
            must["ln_prep_kernel"] = (1, None)
    if p["fused_head"]:
        # head: model.cu:704-705 (ray-layout rows are read as 32-channel segments at stride 64 unless the planes are channel-
        # permuted, model.cu:871-872), model.cu:632 + 711-714 (planes are read directly), io_kernels.cu:447 (instantiation)
        stride = 64 if (p["ray_layout"] == "interleave" and not p["perm"]) else 32
        E = p["E"]
        nk = f"9, {stride}, 17" if E == 544 else ("9, 0, 0" if E > 320 else "5, 0, 0")
        must[f"head_block_kernel<{nk}, {'true' if p['ln_fused'] else 'false'}>"] = (1, 256)
    else:
        # model.cu:732-773: LayerNorm / view mean or Linear / (BN-folded) Linear chain on the fp32 tokens
        never += ["head_block_kernel", "head_fused_kernel"]
    return must, never


def _normalise(name):
    return name.replace("(bool)1", "true").replace("(bool)0", "false")


def traced_forward(m, batch, tmp_path, packed=False):
    """Outputs of one forward and [(kernel name, block.x)] of every kernel it launched (graph_batch=0: no graph replay)."""
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = run_module(m, batch, packed=packed)
    path = tmp_path / "trace.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    kernels = [(_normalise(e["name"]), (e.get("args", {}).get("block") or [None])[0])
               for e in events if e.get("cat") == "kernel"]
    assert kernels, "the trace holds no kernel events"
    return out, kernels


def check_kernels(kernels, must, never, label):
    """Assert `must` ran (launch count, block.x) and nothing of `never` did; returns the "ran" string of the test logs."""
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
