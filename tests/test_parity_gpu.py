"""Parity of the CUDA path (through the nn.Module boundary and the C ABI) against the goldens minted from the
unmodified reference and against the oracle on the same seeded inputs.  Run on the B200 box with `-m gpu`."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from gpu_util import DMPJPE_MM, TOL, build_module, mpjpe_mm, oracle_outputs, rel_err, run_module
from oracle.cases import CASES, make_inputs
from openmpl_b200 import _lib, spec, synth

pytestmark = pytest.mark.gpu

TC_CASES = [n for n in CASES if not CASES[n]["kw"].get("no_transformer_fpt")]


def _check_case(name, precision, packed=False):
    case = CASES[name]
    g = load_golden(name)
    cfg, weights, batch = make_inputs(case)
    m = build_module(case["kw"], weights, precision)
    outs = run_module(m, batch, packed=packed)
    assert m.last_launches > 0
    n_out = 3 if case["kw"].get("head_kadkhod") else 1
    assert len(outs) == n_out
    for i, o in enumerate(outs):
        ref = g[f"out64_{i}"]
        assert o.shape == ref.shape and o.dtype == np.float32
        e = rel_err(o, ref)
        assert e <= TOL[precision], f"{name} [{precision}] out{i}: {e:.3e} of scale"
    d = abs(mpjpe_mm(outs[0], batch["target"].astype(np.float64)) - mpjpe_mm(g["out64_0"], batch["target"].astype(np.float64)))
    assert d <= DMPJPE_MM[precision], f"{name} [{precision}] dMPJPE {d:.4f} mm"
    return outs


@pytest.mark.parametrize("name", list(CASES))
def test_fp32_path_matches_reference_goldens(name):
    _check_case(name, "fp32")


@pytest.mark.parametrize("name", TC_CASES)
def test_tf32_path_matches_reference_goldens(name):
    _check_case(name, "tf32")


@pytest.mark.parametrize("name", TC_CASES)
def test_bf16_path_matches_reference_goldens(name):
    _check_case(name, "bf16")


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_packed_and_list_inputs_agree_bitwise(precision):
    for name in ("flag_hm0flags_small", "cmu0_v2_d2"):
        a = _check_case(name, precision, packed=False)
        b = _check_case(name, precision, packed=True)
        np.testing.assert_array_equal(a[0], b[0])


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
def test_chunking_ragged_and_empty_batches(precision):
    """Arbitrary B: the last chunk is ragged, B = 1 and B = 0 work, and chunking never changes a pose's result."""
    case = CASES["flag_hm0flags_small"]
    cfg = spec.make_config(**case["kw"])
    weights = synth.named_weights(spec.param_spec(cfg), seed=3)
    rig = synth.make_rig(cfg.V)
    batch = synth.make_batch(37, rig, seed=11)
    m = build_module(case["kw"], weights, precision)
    full = run_module(m, batch)[0]
    ref = oracle_outputs(cfg, weights, batch)[0]
    assert rel_err(full, ref) <= TOL[precision]
    m.set_chunk_poses(8)                                           # 37 = 4 * 8 + 5
    chunked = run_module(m, batch)[0]
    np.testing.assert_array_equal(chunked, full)
    one = run_module(m, {k: v[5:6] for k, v in batch.items()})[0]
    np.testing.assert_array_equal(one[0], full[5])
    empty = run_module(m, {k: v[:0] for k, v in batch.items()})[0]
    assert empty.shape == (0, 17, 3)


def test_cpu_inputs_are_accepted_and_output_is_on_the_device():
    case = CASES["flag_conf3rd"]
    cfg, weights, batch = make_inputs(case)
    m = build_module(case["kw"], weights, "fp32")
    V = cfg.V
    args = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])) for v in range(V)] for k in ("poses", "rays", "centers")]
    out = m(args[0], rays=args[1], centers=args[2])
    assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()
    assert rel_err(out.cpu().numpy(), load_golden("flag_conf3rd")["out64_0"]) <= TOL["fp32"]


def test_weights_are_repacked_after_load_state_dict():
    case = CASES["flag_learn3d"]
    cfg, weights, batch = make_inputs(case)
    m = build_module(case["kw"], weights, "fp32")
    a = run_module(m, batch)[0]
    w2 = synth.named_weights(spec.param_spec(cfg), seed=99)
    m.load_state_dict({k: torch.from_numpy(v) for k, v in w2.items()})
    b = run_module(m, batch)[0]
    ref = oracle_outputs(cfg, w2, batch)[0]
    assert rel_err(b, ref) <= TOL["fp32"] and rel_err(a, ref) > 1e-2


def test_data_writes_need_invalidate_and_get_it_from_the_helpers():
    """Writes through `p.data` bump nothing PyTorch exposes: the packed blob stays until `invalidate()` (ADVICE r1);
    `load_state_dict` and `dist.broadcast_state` invalidate on their own."""
    case = CASES["flag_learn3d"]
    cfg, weights, batch = make_inputs(case)
    m = build_module(case["kw"], weights, "fp32")
    a = run_module(m, batch)[0]
    w2 = synth.named_weights(spec.param_spec(cfg), seed=123)
    with torch.no_grad():
        for k, p in m.state_dict(keep_vars=True).items():
            p.data.copy_(torch.from_numpy(w2[k]).to(p.device))          # invisible to the version counter
    stale = run_module(m, batch)[0]
    np.testing.assert_array_equal(stale, a)                              # documented behaviour: still the old weights
    m.invalidate()
    fresh = run_module(m, batch)[0]
    ref = oracle_outputs(cfg, w2, batch)[0]
    assert rel_err(fresh, ref) <= TOL["fp32"] and rel_err(a, ref) > 1e-2


@pytest.mark.parametrize("precision,name,B", [("bf16", "hm0_v4_d12", 2048), ("tf32", "hm0_v4_d12", 1024),
                                             ("bf16", "chosen_v4_d12", 4096), ("bf16", "kptok_v4_d12", 2048),
                                             ("bf16", "cmu_v5_d2_hm0flags", 3000)])
def test_large_batch_pose_independence_against_oracle(precision, name, B):
    """Size-independent property: a pose's output does not depend on the batch around it.  A few hundred poses
    sampled from a large forward (several GEMM tiles, ragged tile tails) are checked against the oracle."""
    case = CASES[name]
    cfg = spec.make_config(**case["kw"])
    weights = synth.named_weights(spec.param_spec(cfg), seed=case["wseed"])
    rig = synth.make_rig(cfg.V, case["rig"])
    batch = synth.make_batch(B, rig, seed=42)
    m = build_module(case["kw"], weights, precision)
    out = run_module(m, batch, packed=True)[0]
    assert np.isfinite(out).all()
    idx = np.unique(np.concatenate([np.arange(8), np.arange(B - 8, B), np.random.default_rng(0).choice(B, 48, replace=False)]))
    sub = {k: v[idx] for k, v in batch.items()}
    ref = oracle_outputs(cfg, weights, sub)[0]
    e = rel_err(out[idx], ref)
    assert e <= TOL[precision], f"{name} [{precision}] B={B}: {e:.3e}"
    d = abs(mpjpe_mm(out[idx], sub["target"].astype(np.float64)) - mpjpe_mm(ref, sub["target"].astype(np.float64)))
    assert d <= DMPJPE_MM[precision]
    # and the same poses alone give the same numbers (bitwise: every kernel is row-independent)
    alone = run_module(m, sub, packed=True)[0]
    np.testing.assert_array_equal(alone, out[idx])


_FUSED_SPT_KW = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=3, num_views=3, drop_path_rate=0.1)


@pytest.mark.parametrize("flags", [
    dict(confidence_as_attention_uncertainty_weight=True, multiple_spatial_blocks=True, confidence_input_as_third=True),
    dict(confidence_as_attention_uncertainty_weight=True, pose_3d_emb_learnable=True),
    dict(qkv_bias=False, qk_scale=0.3, pose_3d_emb_learnable=True),
    dict(add_confidence_input=True, mult_confidence_emb=True, no_transformer_fpt=True),
    dict(depth=1, input_rays_as_token=True),
    dict(confidence_in_FPT=True, input_rays_as_token=True, add_3D_pos_encoding_to_rays=True, multiple_spatial_blocks=True),
    dict(add_3D_pos_encoding_in_Spatial=True, pose_3d_emb_learnable=True, confidence_in_FPT=True),
    dict(add_3D_pos_encoding_in_Spatial=True, input_rays_as_token=True, add_3D_pos_encoding_to_rays=True),
    dict(FPT_blocks_view_keypoint_tokens=True, confidence_input_as_third=True),
], ids=["confattn_multi", "confattn_single", "noqkvbias_scale", "spt_only", "depth1_raytok", "conffpt_interleave",
        "pos3d_spatial_learn", "pos3d_spatial_linear", "kptok_linearpos"])
@pytest.mark.parametrize("B", [5, 77])
def test_fused_spt_kernel_variants_against_oracle(flags, B):
    """The single-kernel SPT (bf16 mode, d = 32, H = 8, J = 17) under the constructor flags that change what it does:
    the confidence-weighted extra pass per block (multiview_mpl.py:406-407), shared vs per-view stacks, no qkv bias,
    explicit qk_scale, depth 1 (the only block runs twice), batches that do not fill a CTA tile, and every variant of
    the joint embedding fused into its prologue (confidence add / mult, learnable 3D position; the ray-direction
    position falls back to the separate embed kernel) and of the token build fused into its epilogue (three ray
    layouts, confidence-in-FPT, table vs Linear(normalize(ray)) position codes)."""
    kw = dict(_FUSED_SPT_KW, **flags)
    cfg = spec.make_config(**kw)
    weights = synth.named_weights(spec.param_spec(cfg), seed=5)
    batch = synth.make_batch(B, synth.make_rig(cfg.V), seed=9)
    m = build_module(kw, weights, "bf16")
    out = run_module(m, batch)[0]
    ref = oracle_outputs(cfg, weights, batch)[0]
    e = rel_err(out, ref)
    assert e <= TOL["bf16"], f"{flags}: {e:.3e} of scale"


@pytest.mark.parametrize("name", ["hm0_v4_d12", "chosen_v4_d12", "cmu_v5_d2_hm0flags", "sweep_viewtok_v3", "flag_depth1"])
def test_layernorm_fusion_on_and_off_agree_with_the_reference(name):
    """bf16 mode folds the FPT LayerNorms into the projection GEMMs (rank-1 form, DESIGN.md §4); the unfused form
    (separate LayerNorm kernels) stays selectable.  Both must meet the bf16 bound and agree with each other closely."""
    case = CASES[name]
    g = load_golden(name)
    cfg, weights, batch = make_inputs(case)
    outs = {}
    for fused in (1, 0):
        m = build_module(case["kw"], weights, "bf16", ln_fusion=bool(fused))
        outs[fused] = run_module(m, batch)[0]
        assert rel_err(outs[fused], g["out64_0"]) <= TOL["bf16"]
    assert rel_err(outs[1], outs[0].astype(np.float64)) <= TOL["bf16"]


@pytest.mark.parametrize("precision", ["fp32", "tf32", "bf16"])
def test_cuda_graph_small_batch_path_equals_the_plain_path(precision):
    """Batches up to `graph_batch` poses (the reference runner's TEST.BATCH_SIZE = 256) are captured once per batch size as a
    CUDA graph and replayed: same numbers as the kernel-by-kernel path, one capture, then replays -- also for fresh input
    tensors at new addresses (the module stages them in persistent buffers), host tensors and the packed layout."""
    case = CASES["flag_hm0flags_small"]
    cfg = spec.make_config(**case["kw"])
    weights = synth.named_weights(spec.param_spec(cfg), seed=3)
    rig = synth.make_rig(cfg.V)
    plain = build_module(case["kw"], weights, precision, graph_batch=0)
    graph = build_module(case["kw"], weights, precision, graph_batch=512)
    outs = []
    for seed in (1, 2, 3):
        batch = synth.make_batch(256, rig, seed=seed)
        a = run_module(plain, batch)[0]
        b = run_module(graph, batch)[0]
        np.testing.assert_array_equal(a, b)
        outs.append(b)
    assert not np.array_equal(outs[0], outs[1])                       # the replays really consumed the new inputs
    assert plain.graph_stats() == (0, 0)
    assert graph.graph_stats() == (1, 2)
    batch = synth.make_batch(256, rig, seed=4)
    np.testing.assert_array_equal(run_module(graph, batch, packed=True)[0], run_module(plain, batch)[0])   # second layout: second graph
    V = cfg.V
    host = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])) for v in range(V)] for k in ("poses", "rays", "centers")]
    with torch.no_grad():
        out = graph(host[0], rays=host[1], centers=host[2])
    torch.cuda.synchronize()
    np.testing.assert_array_equal(out.cpu().numpy(), run_module(plain, batch)[0])
    big = synth.make_batch(600, rig, seed=5)                          # above graph_batch: plain path, no new capture
    caps = graph.graph_stats()[0]
    np.testing.assert_array_equal(run_module(graph, big)[0], run_module(plain, big)[0])
    assert graph.graph_stats()[0] == caps
    assert rel_err(outs[0], oracle_outputs(cfg, weights, synth.make_batch(256, rig, seed=1))[0]) <= TOL[precision]


@pytest.mark.parametrize("name", ["hm0_v4_d12", "cmu0_v2_d2", "sweep_viewtok_v8", "sweep_viewtok_v2", "cmu_v5_d2_hm0flags",
                                  "sweep_viewtok_v3", "sweep_viewtok_v5", "sweep_viewtok_v6", "sweep_viewtok_v7",
                                  "chosen_v4_d12", "cmu_v5_d2_chosen"])
def test_fused_qkv_attention_on_and_off_agree_with_the_reference(name):
    """bf16 mode runs the QKV projection and the cross-view attention as ONE kernel for 2 to 8 views of 136- or 68-wide heads (no
    q|k|v tensor); the two-kernel form stays selectable (`qkv_attn_fusion=False`) and serves every other shape.  Both must
    meet the bf16 bound against the reference goldens and agree with each other; a large batch covers many tiles per CTA."""
    case = CASES[name]
    g = load_golden(name)
    cfg, weights, batch = make_inputs(case)
    outs = {}
    for fused in (True, False):
        m = build_module(case["kw"], weights, "bf16", qkv_attn_fusion=fused)
        outs[fused] = run_module(m, batch)[0]
        assert rel_err(outs[fused], g["out64_0"]) <= TOL["bf16"]
    assert rel_err(outs[True], outs[False].astype(np.float64)) <= TOL["bf16"]
    big = synth.make_batch(3000, synth.make_rig(cfg.V, case["rig"]), seed=77)
    a = run_module(build_module(case["kw"], weights, "bf16", qkv_attn_fusion=True), big, packed=True)[0]
    b = run_module(build_module(case["kw"], weights, "bf16", qkv_attn_fusion=False), big, packed=True)[0]
    assert np.isfinite(a).all() and rel_err(a, b.astype(np.float64)) <= TOL["bf16"]


def test_native_library_is_what_ran():
    _lib.lib()                                    # (a no-op after any forward; keeps the test order independent)
    maps = open("/proc/self/maps").read()
    assert "libmpl_b200.so" in maps


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_data_parallel_replicas_like_the_reference_runner(precision):
    """The reference's only multi-GPU mechanism: `torch.nn.DataParallel(model, device_ids=gpus).cuda()` fed lists of
    CPU tensors (MPL/run/valid_mpl.py:177-178, core/function_mpl.py:344-350).  Replicas share the C handle and keep
    per-device packed weights; the gathered output must equal the single-GPU output."""
    case = CASES["cmu0_v2_d2"]
    cfg, weights, _ = make_inputs(case)
    batch = synth.make_batch(64, synth.make_rig(cfg.V, "cmu"), seed=3)
    m = build_module(case["kw"], weights, precision)
    single = run_module(m, batch)[0]
    dp = torch.nn.DataParallel(m, device_ids=[0, 1]).cuda()
    V = cfg.V
    args = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])) for v in range(V)] for k in ("poses", "rays", "centers")]
    with torch.no_grad():
        out = dp(args[0], rays=args[1], centers=args[2])
    torch.cuda.synchronize()
    assert out.shape == (64, 17, 3) and out.device.index == 0
    np.testing.assert_array_equal(out.cpu().numpy(), single)


@pytest.mark.parametrize("packed,first", [(False, None), (True, None), (True, 100), (False, 7)])
def test_pipelined_host_staging_equals_device_resident_inputs(packed, first):
    """Host inputs spanning several forward chunks take the pipelined path (copy of chunk i+1 overlapped with the compute
    of chunk i on a side stream); the result must be bitwise the result of the same call on device-resident inputs."""
    case = CASES["cmu0_v2_d2"]
    cfg, weights, _ = make_inputs(case)
    batch = synth.make_batch(1000, synth.make_rig(cfg.V, "cmu"), seed=12)
    m = build_module(case["kw"], weights, "bf16")
    m.set_chunk_poses(256)                                           # 1000 = 3 * 256 + 232
    if first is not None:
        m.pipeline_first_poses = first                               # a short, unaligned first piece: 1000 = 100 + 3 * 256 + 132
    ref = run_module(m, batch, packed=packed)[0]                     # device-resident inputs
    V = cfg.V
    if packed:
        args = [torch.from_numpy(batch[k]).pin_memory() for k in ("poses", "rays", "centers")]
    else:
        args = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])).pin_memory() for v in range(V)]
                for k in ("poses", "rays", "centers")]
    with torch.no_grad():
        out = m(args[0], rays=args[1], centers=args[2])
    torch.cuda.synchronize()
    np.testing.assert_array_equal(out.cpu().numpy(), ref)
    assert m.last_launches > 0
