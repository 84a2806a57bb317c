"""The constructor-flag matrix at production width (d = 32, H = 8, J = 17, depth 2): every flag case of the goldens
(oracle/cases.py, built there at d = 16, H = 4) except the J = 13 one, plus the `hm_0` flag set with each non-default
head, with the confidence-weighted SPT and with MLP ratio 3, and the keypoint-token set with the confidence as a third
input channel.  Shared by test_flag_paths_gpu.py (forward against the oracle, kernel path) and test_flag_paths_cpu.py
(every flag is in the matrix, every case is a valid configuration)."""
from collections import OrderedDict

from oracle.cases import _FLAG_CASES
from openmpl_b200 import spec

PROD = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=2, drop_rate=0.0, attn_drop_rate=0.0, drop_path_rate=0.1)
KPTOK_FLAGS = dict(pose_3d_emb_learnable=True, FPT_blocks_view_keypoint_tokens=True)   # the goldens' keypoint-token set

FLAG_CASES = OrderedDict((n, dict(f)) for n, f in _FLAG_CASES.items() if n != "j13")   # J = 13: test_view_counts_gpu.py
FLAG_CASES["hm0flags_deephead"] = dict(spec.HM0_FLAGS, deep_head=True)
FLAG_CASES["hm0flags_kadkhod"] = dict(spec.HM0_FLAGS, head_kadkhod=True)
FLAG_CASES["hm0flags_linmean"] = dict(spec.HM0_FLAGS, linear_weighted_mean=True)
FLAG_CASES["hm0flags_confattn"] = dict(spec.HM0_FLAGS, confidence_as_attention_uncertainty_weight=True)
FLAG_CASES["hm0flags_mlp3"] = dict(spec.HM0_FLAGS, mlp_ratio=3.0)
FLAG_CASES["kptok_conf3rd"] = dict(KPTOK_FLAGS, confidence_input_as_third=True)

# golden-pinned architecture of each FPT kind: the bf16 sibling of a case (same seeds, batch and V)
SIBLINGS = {"chosen": dict(spec.CHOSEN_FLAGS), "hm0": dict(spec.HM0_FLAGS), "kptok": dict(KPTOK_FLAGS)}


def case_kw(name, V):
    return dict(PROD, **FLAG_CASES[name], num_views=V)


def sibling_of(name, V=4):
    """"kptok" for keypoint tokens, "hm0" for D = 1088 view tokens (rays as tokens), "chosen" for D = 544."""
    cfg = spec.make_config(**case_kw(name, V))
    if cfg.kw["FPT_blocks_view_keypoint_tokens"]:
        return "kptok"
    return "hm0" if cfg.tok_w == 2 * cfg.E else "chosen"


def views_of(name):
    """V = 4 for every case; also V = 5 where the FPT runs on D = 544 / 1088 view tokens: at V = 5 the fused QKV + attention
    kernel tiles its rows pose-aligned instead of 128-aligned (gemm_tcgen05.cu qkv_attn_kernel)."""
    cfg = spec.make_config(**case_kw(name, 4))
    fpt_views = not cfg.kw["no_transformer_fpt"] and not cfg.kw["FPT_blocks_view_keypoint_tokens"]
    return [4, 5] if fpt_views and cfg.fpt_dim in (544, 1088) else [4]
