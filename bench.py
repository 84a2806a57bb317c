#!/usr/bin/env python
"""bench.py — poses/s of the MPL lifter forward (BASELINE.json metric) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision bf16|tf32|fp32]
                    [--arch hm0|chosen|cmu0|kptok] [--views V] [--depth D] [--batch B] [--dump-outputs DIR]

One "step" = one forward of the H36M 4-view 17-joint `hm_0` lifter (depth 12, D = 1088, 114 M parameters) over a
batch of 65 536 synthetic poses per GPU (BASELINE.json configs[1]).  Ranks shard the pose index range; there is no
data-path collective, only one all-reduce of the MPJPE accumulators after the timed region.  Prints ONE JSON line.
`--arch / --views / --depth` select the other BASELINE.json configurations (CMU Panoptic V = 5 depth 2, the "chosen"
ablation, the view sweep in both token layouts) with the same keys.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "poses/sec MPL forward (H36M 4-view, 17 joints)"
ARCH = dict(num_joints=17, embed_dim_ratio=32, num_heads=8, depth=12, num_views=4, drop_path_rate=0.1)
ARCH_NAMES = {"hm0": "H36M hm_0 (MultiSPT, Conf3rd, Raytoken, Add3dEncRays)", "cmu0": "CMU Panoptic cmu_0 flags (= hm_0 flags)",
              "chosen": "'chosen' ablation (single SPT, no ray token)", "kptok": "view x keypoint-token FPT"}
ARCH_DEPTH = {"hm0": 12, "chosen": 12, "kptok": 12, "cmu0": 2}
ARCH_VIEWS = {"hm0": 4, "chosen": 4, "kptok": 4, "cmu0": 5}
ARCH_RIG = {"hm0": "h36m", "chosen": "h36m", "kptok": "h36m", "cmu0": "cmu"}
DUMP_LIMIT = 64 << 20          # bytes written by --dump-outputs at most


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    p.add_argument("--precision", default=os.environ.get("MPL_BENCH_PRECISION", "bf16"), choices=["bf16", "tf32", "fp32"])
    p.add_argument("--batch", type=int, default=65536, help="poses per GPU per step")
    p.add_argument("--cpu-batch", type=int, default=1024, help="poses per CPU-baseline forward")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--arch", default="hm0", choices=sorted(ARCH_NAMES))
    p.add_argument("--views", type=int, default=None)
    p.add_argument("--depth", type=int, default=None)
    p.add_argument("--parity-poses", type=int, default=512, help="poses of the step checked against the oracle (outside the timed regions)")
    p.add_argument("--no-extras", action="store_true", help="skip the latency_b256 and fp32-grade-mode side measurements")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the output of the last timed step to DIR/output.npy (float32, rank 0's shard; above "
                        f"{DUMP_LIMIT >> 20} MB a fixed seeded sample of its poses) so that two builds can be compared")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs applies to --impl ours")
    a.views = a.views or ARCH_VIEWS[a.arch]
    a.depth = ARCH_DEPTH[a.arch] if a.depth is None else a.depth
    return a


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def workload(args):
    from openmpl_b200 import spec
    flags = {"hm0": spec.HM0_FLAGS, "cmu0": spec.HM0_FLAGS, "chosen": spec.CHOSEN_FLAGS,
             "kptok": dict(pose_3d_emb_learnable=True, confidence_input_as_third=True, FPT_blocks_view_keypoint_tokens=True)}[args.arch]
    kw = dict(ARCH, depth=args.depth, num_views=args.views, **flags)
    return kw, spec.make_config(**kw)


def metric_name(args):
    if args.arch == "hm0" and args.views == 4:
        return METRIC
    rig = "H36M" if ARCH_RIG[args.arch] == "h36m" else "CMU Panoptic"
    return f"poses/sec MPL forward ({rig} {args.views}-view, 17 joints)"


def workload_name(args, cfg, batch, what):
    rig = "H36M" if ARCH_RIG[args.arch] == "h36m" else "CMU Panoptic"
    return (f"{rig} {cfg.V}-view 17-joint lifter forward, {ARCH_NAMES[args.arch]}, depth {cfg.depth}, D={cfg.fpt_dim}, "
            f"{cfg.fpt_tokens} FPT tokens, {what}")


def cpu_forward_timer(args, steps, warmup):
    """The reference forward timed on the host cores, fp32, all cores.  kind "reference": the UNMODIFIED reference module
    (`MPL/lib/models/multiview_mpl.py`, staged byte for byte under the git-ignored oracle/_ref/ by oracle/stage_reference.py)
    run through its own forward; kind "port" (only when the staged file is missing): the torch-CPU restatement making the
    same ATen calls.  Returns (per-forward seconds, kind)."""
    import torch
    from openmpl_b200 import spec, synth
    from oracle import ref_loader                                   # cpu_baseline / --impl reference legs only
    torch.set_num_threads(os.cpu_count() or 1)
    kw, cfg = workload(args)
    batch = synth.make_batch(args.cpu_batch, synth.make_rig(cfg.V, ARCH_RIG[args.arch]), seed=1)
    V = cfg.V
    if ref_loader.model_file() is not None:
        kind = "reference"
        mod = ref_loader.load_model_module()
        torch.manual_seed(0)
        model = mod.MultiView_MPL(**kw).eval()                      # PyTorch default init under seed 0 = the reference's 'scratch' init
        lists = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])) for v in range(V)] for k in ("poses", "rays", "centers")]

        def fwd():
            with torch.no_grad():
                return model(lists[0], rays=lists[1], centers=lists[2])
    else:
        kind = "port"
        from oracle import torch_port
        weights = synth.named_weights(spec.param_spec(cfg), seed=0)
        p = {k: torch.from_numpy(v) for k, v in weights.items()}
        x = [torch.from_numpy(batch[k]) for k in ("poses", "rays", "centers")]
        fwd = lambda: torch_port.forward(p, cfg, *x)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        fwd()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return times, kind


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path (the unmodified module when staged, see
    cpu_forward_timer) on all host cores; each step = one forward over a bounded sample of the workload."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    steps, warmup = args.steps, max(1, min(args.warmup, 5))   # K timed forwards, W untimed
    times, kind = cpu_forward_timer(args, steps, warmup)
    total = sum(times)
    value = args.cpu_batch * len(times) / total
    kw, cfg = workload(args)
    what = ("the unmodified reference module (MPL/lib/models/multiview_mpl.py) through its own forward" if kind == "reference"
            else "torch-CPU fp32 restatement of MultiView_MPL.forward (same ATen calls as the reference)")
    line = {
        "impl": "reference", "metric": metric_name(args), "value": value, "unit": "poses/s", "n_gpus": args.gpus, "steps": len(times),
        "warmup": warmup, "ms_per_step": 1000.0 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args, cfg, args.batch, f"batch {args.batch} per GPU"),
                   "sample": f"bounded sample of {args.cpu_batch} poses per step", "batch_per_step": args.cpu_batch,
                   "views": cfg.V, "joints": cfg.J, "note": what + ", all host cores"},
        "cpu_baseline": {"value": value, "unit": "poses/s", "cores": cores, "kind": kind,
                         "sample": f"{len(times)} forwards of {args.cpu_batch} poses"},
        "e2e": {"value": value, "unit": "poses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_reference_gpu(args):
    """--impl reference-gpu: the second comparator of SURVEY.md section 8d -- the UNMODIFIED reference module (staged under
    oracle/_ref/) run as PyTorch-eager library kernels (cuBLAS / ATen; the reference ships no GPU kernels of its own) on
    cuda:0, CUDA-event timed, at its runner's own batch (256) and at the bench batch: fp32 (TF32 off), TF32 allowed, bf16
    autocast.  `value` is the most favourable of them at the bench batch."""
    import contextlib
    import torch
    from openmpl_b200 import synth
    from oracle import ref_loader                                   # reference arm only
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if ref_loader.model_file() is None or not torch.cuda.is_available():
        print(json.dumps({"impl": "reference-gpu", "unavailable": "needs the staged reference module (oracle/_ref) and a GPU"}), flush=True)
        return
    kw, cfg = workload(args)
    mod = ref_loader.load_model_module()
    torch.manual_seed(0)
    dev = torch.device("cuda", 0)
    model = mod.MultiView_MPL(**kw).eval().to(dev)
    V = cfg.V
    steps, warmup = args.steps, max(2, min(args.warmup, 5))
    modes = {}
    for B in sorted({256, args.batch}):
        batch = synth.make_batch(B, synth.make_rig(V, ARCH_RIG[args.arch]), seed=1)
        lists = [[torch.from_numpy(np.ascontiguousarray(batch[k][:, v])).to(dev) for v in range(V)] for k in ("poses", "rays", "centers")]
        for mode in ("fp32", "tf32", "bf16_autocast"):
            torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = mode == "tf32"
            ctx = torch.autocast("cuda", dtype=torch.bfloat16) if mode == "bf16_autocast" else contextlib.nullcontext()
            with torch.no_grad(), ctx:
                for _ in range(warmup):
                    model(lists[0], rays=lists[1], centers=lists[2])
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(steps):
                    model(lists[0], rays=lists[1], centers=lists[2])
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            modes[f"{mode}_b{B}"] = {"poses_per_s": B / (ms / 1e3), "ms_per_forward": ms}
    best = max(("fp32", "tf32", "bf16_autocast"), key=lambda m: modes[f"{m}_b{args.batch}"]["poses_per_s"])
    line = {"impl": "reference-gpu", "metric": metric_name(args), "value": modes[f"{best}_b{args.batch}"]["poses_per_s"], "unit": "poses/s",
            "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": modes[f"{best}_b{args.batch}"]["ms_per_forward"],
            "higher_is_better": True, "dtype": best, "data": "synthetic",
            "config": {"workload": workload_name(args, cfg, args.batch, f"batch {args.batch} per GPU"),
                       "note": "the unmodified reference module (MPL/lib/models/multiview_mpl.py) as PyTorch-eager library kernels on cuda:0, "
                               "inputs resident on the device; not the tier's reference arm (that is --impl reference, host cores)"},
            "modes": modes, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.f.read().strip().splitlines():
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.f.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        # median over the samples taken under load (upper half of the power readings)
        order = np.argsort(pw)[len(pw) // 2:]
        return {"sm_mhz": float(np.median(np.asarray(sm)[order])), "sm_max_mhz": float(max(mx)),
                "power_w_max": float(max(pw)), "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir, out):
    """Write a step's output (B, J, 3) to out_dir/output.npy; above DUMP_LIMIT bytes, the rows of a fixed seeded sample of
    poses (in index order), so that runs with the same arguments write the same poses."""
    host = out.cpu().numpy()
    rows = len(host)
    if host.nbytes > DUMP_LIMIT:
        keep = DUMP_LIMIT // host[0].nbytes
        host = host[np.sort(np.random.default_rng(0).choice(rows, size=keep, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, "output.npy")
    np.save(path, host)
    return {"file": path, "shape": list(host.shape), "poses_of": rows,
            "sample": None if len(host) == rows else "numpy default_rng(0).choice without replacement, sorted"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from openmpl_b200 import _lib, dist as mdist, metric, spec, synth
    from openmpl_b200.models.multiview_mpl_b200 import MultiView_MPL

    rank, world, local = mdist.init_from_env("nccl")
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}", file=sys.stderr)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    kw, cfg = workload(args)
    B = args.batch
    pk, pk_src = peaks()

    # ---- model: random-init weights of the named architecture (seeded, identical on every rank) ----
    weights = synth.named_weights(spec.param_spec(cfg), seed=0)
    impl = {}
    if os.environ.get("MPL_GEMM_CTA_GROUP"):
        impl["gemm_cta_group"] = int(os.environ["MPL_GEMM_CTA_GROUP"])
    if os.environ.get("MPL_LN_FUSION"):
        impl["ln_fusion"] = bool(int(os.environ["MPL_LN_FUSION"]))
    if os.environ.get("MPL_QKV_ATTN_FUSION"):
        impl["qkv_attn_fusion"] = bool(int(os.environ["MPL_QKV_ATTN_FUSION"]))
    if os.environ.get("MPL_CHUNK_STREAMS"):
        impl["chunk_streams"] = int(os.environ["MPL_CHUNK_STREAMS"])
    model = MultiView_MPL(**kw, precision=args.precision, **impl)
    model.load_state_dict({k: torch.from_numpy(v) for k, v in weights.items()})
    model = model.to(dev).eval()
    if os.environ.get("MPL_CHUNK"):
        model.set_chunk_poses(int(os.environ["MPL_CHUNK"]))

    # ---- synthetic inputs of this rank's shard of the global pose range ----
    start, _ = mdist.shard_range(B * world, rank, world)
    rig = synth.make_rig(cfg.V, ARCH_RIG[args.arch])
    batch = synth.make_batch(B, rig, seed=1, start=start)
    host = {k: torch.from_numpy(batch[k]).pin_memory() for k in ("poses", "rays", "centers", "target")}
    devin = {k: v.to(dev) for k, v in host.items()}
    h2d = world * sum(host[k].numel() * 4 for k in ("poses", "rays", "centers"))     # whole job, all ranks
    d2h = world * B * cfg.J * 3 * 4

    def step_device():
        with torch.no_grad():
            return model(devin["poses"], rays=devin["rays"], centers=devin["centers"])

    host_out = torch.empty((B, cfg.J, 3), dtype=torch.float32).pin_memory()

    def step_e2e():
        with torch.no_grad():
            out = model(host["poses"], rays=host["rays"], centers=host["centers"])     # H2D inside the module call
        host_out.copy_(out, non_blocking=True)                                          # D2H of the step's result (pinned)
        torch.cuda.synchronize()
        return host_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- parity against the oracle (checker only; outside every timed region): poses spread over the whole batch, i.e.
    # over every forward chunk and many GEMM tiles ----
    out = step_device()
    parity = None
    if rank == 0 and args.parity_poses > 0:
        from oracle import mpl_oracle
        n = min(args.parity_poses, B)
        idx = np.unique(np.linspace(0, B - 1, n).astype(np.int64))
        ref = mpl_oracle.forward(weights, cfg, batch["poses"][idx], batch["rays"][idx], batch["centers"][idx])
        got = out[torch.from_numpy(idx).to(dev)].cpu().numpy()
        scale = float(np.abs(ref).max())
        tgt = batch["target"][idx].astype(np.float64)
        mp = lambda p: float(np.sqrt(((p - tgt) ** 2).sum(-1)).mean()) * 1000.0
        chunk0 = int(model.chunk_poses())
        parity = {"max_abs_err_over_scale": float(np.abs(got - ref).max()) / scale, "poses_checked": int(len(idx)),
                  "chunks_covered": int(len(np.unique(idx // chunk0))), "delta_mpjpe_mm": abs(mp(got.astype(np.float64)) - mp(ref)),
                  "stated_bound": {"bf16": 1.2e-2, "tf32": 1e-3, "fp32": 2e-5}[args.precision]}

    # ---- timed region 1: device-resident inputs (value) ----
    for _ in range(max(args.warmup, 3)):
        step_device()
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    e0.record()
    for _ in range(args.steps):
        last = step_device()
        launches += model.last_launches
    e1.record()
    barrier()
    ms = mdist.max_over_ranks(e0.elapsed_time(e1), dev)
    clocks = sampler.stop() if sampler else None
    value = world * args.steps * B / (ms / 1000.0)
    dump = dict(dump_outputs(args.dump_outputs, last), ranks=[0], world_size=world) if args.dump_outputs and rank == 0 else None
    del last

    # ---- timed region 2: end to end through the module call with host buffers (e2e) ----
    for _ in range(2):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    torch.cuda.synchronize()
    ms_e2e = mdist.max_over_ranks((time.perf_counter() - t0) * 1000.0, dev)
    barrier()
    e2e_value = world * args.steps * B / (ms_e2e / 1000.0)

    # ---- per-kernel breakdown with CUDA events on the launch stream (roofline) ----
    # (chunks serialised while profiling: with two chunks in flight the launches of the two streams interleave on the SMs and an
    # event pair around one launch would also time its wait for the other stream's kernel)
    model.set_profile(True, serial=True)
    prof_steps = 2
    agg = {}
    for _ in range(prof_steps):
        step_device()
        for k, (t, n) in model.profile().items():
            a = agg.setdefault(k, [0.0, 0])
            a[0] += t; a[1] += n
    model.set_profile(False)
    gemm_cats = ["fpt_gemm_qkv", "fpt_gemm_proj", "fpt_gemm_fc1", "fpt_gemm_fc2"]
    D, Hf, M = cfg.fpt_dim, cfg.fpt_hidden, B * cfg.fpt_tokens
    flops_per_launch = {"fpt_gemm_qkv": 2.0 * M * 3 * D * D, "fpt_gemm_proj": 2.0 * M * D * D,
                        "fpt_gemm_fc1": 2.0 * M * Hf * D, "fpt_gemm_fc2": 2.0 * M * D * Hf}
    # the last fc2 of the stack computes only the columns the head reads (mpl_dim 7): count what is executed, not the dead half
    n_last = int(_lib.lib().mpl_dim(model._get_handle(), 7)) if args.precision == "bf16" else D
    apps = cfg.depth + 1
    flops_per_launch["fpt_gemm_fc2"] *= (apps - 1 + n_last / D) / apps
    chunk_poses = int(os.environ.get("MPL_CHUNK", "0")) or int(model.chunk_poses())
    chunks = -(-B // chunk_poses)
    roofline, breakdown = None, {}
    try:      # per-launch DRAM traffic of the GEMM launches from the committed `ncu --set full` capture (profiles/)
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(args.arch, {})
    except Exception:
        traffic = {}
    tot_ms = sum(a[0] for a in agg.values())
    for k, (t, n) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
        breakdown[k] = {"ms_per_step": t / prof_steps, "launches_per_step": n // prof_steps, "share": t / tot_ms if tot_ms else 0}
    if all(c in agg for c in gemm_cats):
        g_ms = sum(agg[c][0] for c in gemm_cats)
        g_n = sum(agg[c][1] for c in gemm_cats)
        # algorithmic FLOPs of the launches timed: each category launches (depth+1) * chunks times per step on M / chunks rows
        g_flops = sum(flops_per_launch[c] / chunks * agg[c][1] for c in gemm_cats)
        achieved = g_flops / (g_ms / 1000.0) / 1e12
        # tf32-named mode = split bf16 operands: three bf16 MMAs per algorithmic product
        peak = pk.get("bf16_tflops_sustained", 1400.0) / (3.0 if args.precision == "tf32" else 1.0)
        fused_attn = "fpt_attention" not in agg
        roofline = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel / qkv_attn_kernel (QKV/proj/fc1/fc2 of the FPT)"
                    + ("; the QKV launches are the fused QKV + cross-view-attention kernel: their time includes the attention, "
                       "their FLOPs count the projection only" if fused_attn else ""), "achieved": achieved,
                    "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": traffic.get("gemm_tcgen05_kernel", {}).get("bytes_per_launch"),
                    "traffic_note": traffic.get("gemm_tcgen05_kernel", {}).get("note"),
                    "traffic_capture": {k: traffic.get("gemm_tcgen05_kernel", {}).get(k) for k in ("capture", "git_rev_at_capture", "lib_sha256_16")},
                    "per_gemm_tflops": {c: flops_per_launch[c] / chunks * agg[c][1] / (agg[c][0] / 1000.0) / 1e12 for c in gemm_cats},
                    "algorithmic_flops_per_launch": g_flops / g_n,
                    "peak_source": f"{pk_src} bf16_tflops_sustained" + (" / 3 (split bf16 hi/lo operands)" if args.precision == "tf32" else ""),
                    "avg_launch_ms": g_ms / g_n, "launches_timed": g_n, "share_of_step": g_ms / tot_ms}
    elif agg:
        k = max(agg, key=lambda c: agg[c][0])
        roofline = {"bound": "tensor", "kernel": k, "achieved": None, "peak": None, "unit": "TFLOP/s", "frac": None,
                    "traffic": None, "note": "fp32 CUDA-core path: no tensor-core kernel in this mode"}

    # ---- HBM-bound kernels: algorithmic bytes per launch / measured launch time vs the measured copy bandwidth ----
    Bc = min(B, chunk_poses)
    rows_f = Bc * cfg.fpt_tokens
    esz = 2 if args.precision == "bf16" else 4
    alg_bytes = {
        "embed": Bc * cfg.V * (cfg.J * 12 + cfg.J * cfg.d * 4),
        "token_build": Bc * cfg.V * (cfg.J * cfg.d * 4 + 2 * cfg.J * 12 + 12 + cfg.tok_w * 4),
        "fpt_attention": rows_f * (3 * D + D) * esz,
        # bf16 mode: ln_prep (fp32 tokens -> two bf16 planes), once per chunk; other modes: LayerNorm kernels
        "fpt_layernorm": rows_f * (D * 4 + D * (4 if args.precision != "fp32" else 4)),
        "head": Bc * (cfg.V * cfg.E * 4 + cfg.J * 12),
    }
    memory_kernels = {}
    for k, nbytes in alg_bytes.items():
        if k in agg and agg[k][1]:
            ms_l = agg[k][0] / agg[k][1]
            gbs = nbytes / (ms_l * 1e-3) / 1e9
            memory_kernels[k] = {"avg_launch_ms": ms_l, "algorithmic_bytes_per_launch": nbytes, "achieved_gbs": gbs,
                                 "frac_of_hbm_peak": gbs / pk.get("hbm_gbs", 6650.0)}
            cap = traffic.get("head_block_kernel") if k == "head" else None
            if cap and Bc == 32768 and args.precision == "bf16":
                # what DRAM really moves for this launch (ncu capture of the same chunk size, profiles/ncu_traffic.json)
                dgbs = cap["bytes_per_launch"] / (ms_l * 1e-3) / 1e9
                memory_kernels[k].update({"dram_bytes_per_launch_ncu": cap["bytes_per_launch"], "dram_gbs": dgbs,
                                          "dram_frac_of_hbm_peak": dgbs / pk.get("hbm_gbs", 6650.0),
                                          "ncu_alone": {"launch_ms": cap["ncu_launch_s"] * 1e3, "dram_gbs": cap["ncu_dram_gbs"]}})

    # ---- the collectives: MPJPE / P-MPJPE accumulators all-reduced over ranks (NCCL) ----
    acc = metric.MpjpeAccumulator(cfg.J, output_in_meter=True, device=dev)
    acc.update(out, devin["target"])
    acc.all_reduce()
    res = acc.result()
    pacc = metric.PmpjpeAccumulator(cfg.J, output_in_meter=True, device=dev)
    pacc.update(out, devin["target"])
    pacc.all_reduce()
    pres = pacc.result()

    # ---- CPU baseline (rank 0, N = 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        times, kind = cpu_forward_timer(args, steps=3, warmup=1)
        v = args.cpu_batch * len(times) / sum(times)
        cpu = {"value": v, "unit": "poses/s", "cores": os.cpu_count(), "kind": kind,
               "sample": f"{len(times)} forwards of {args.cpu_batch} poses ("
                         + ("the unmodified reference module" if kind == "reference" else "torch-CPU fp32 restatement of the reference forward")
                         + ", fp32, all cores)"}

    # ---- side measurements (rank 0, N = 1; outside the timed regions above) ----
    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        # (1) the reference runner's own batch size (TEST.BATCH_SIZE 256, lists of host tensors, valid_mpl.py:205-210): end to
        # end through the module, CUDA-graph path vs kernel-by-kernel launches
        b256 = synth.make_batch(256, rig, seed=2)
        lists = [[torch.from_numpy(np.ascontiguousarray(b256[k][:, v])).pin_memory() for v in range(cfg.V)]
                 for k in ("poses", "rays", "centers")]
        lat = {}
        for tag, gb in (("cuda_graph", 2048), ("kernel_by_kernel", 0)):
            m2 = MultiView_MPL(**kw, precision=args.precision, graph_batch=gb, **impl)
            m2.load_state_dict({k: torch.from_numpy(v) for k, v in weights.items()})
            m2 = m2.to(dev).eval()
            res_host = torch.empty((256, cfg.J, 3), dtype=torch.float32).pin_memory()

            def call():
                with torch.no_grad():
                    o = m2(lists[0], rays=lists[1], centers=lists[2])
                res_host.copy_(o, non_blocking=True)
                torch.cuda.synchronize()
            for _ in range(5):
                call()
            t0 = time.perf_counter()
            for _ in range(50):
                call()
            dt = (time.perf_counter() - t0) / 50
            d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            d0.record()
            for _ in range(20):
                call()
            d1.record()
            torch.cuda.synchronize()
            dev_in = [[t.to(dev) for t in ts] for ts in lists]      # device-resident lists: the forward alone
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.no_grad():
                for _ in range(5):
                    m2(dev_in[0], rays=dev_in[1], centers=dev_in[2])
                g0.record()
                for _ in range(20):
                    m2(dev_in[0], rays=dev_in[1], centers=dev_in[2])
                g1.record()
            torch.cuda.synchronize()
            lat[tag] = {"ms": dt * 1e3, "poses_per_s": 256 / dt, "launches": m2.last_launches,
                        "forward_only_device_inputs_ms": g0.elapsed_time(g1) / 20}
            del m2
        extras["latency_b256"] = dict(lat, note="host lists in -> pinned host result out, H2D + D2H inside, mean of 50 calls")
        # (2) the fp32-grade tensor-core mode (split bf16 hi/lo operands) on the same workload: the mode that carries the
        # 1e-3 / 0.1 mm parity bound
        if args.precision == "bf16":
            m3 = MultiView_MPL(**kw, precision="tf32", **impl)
            m3.load_state_dict({k: torch.from_numpy(v) for k, v in weights.items()})
            m3 = m3.to(dev).eval()
            with torch.no_grad():
                o3 = m3(devin["poses"], rays=devin["rays"], centers=devin["centers"])
                for _ in range(2):
                    m3(devin["poses"], rays=devin["rays"], centers=devin["centers"])
                torch.cuda.synchronize()
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
                for _ in range(3):
                    m3(devin["poses"], rays=devin["rays"], centers=devin["centers"])
                a1.record()
                torch.cuda.synchronize()
            ms3 = a0.elapsed_time(a1) / 3
            err3 = None
            if parity is not None:
                got3 = o3[torch.from_numpy(idx).to(dev)].cpu().numpy()
                err3 = float(np.abs(got3 - ref).max()) / scale
            extras["fp32_grade_mode"] = {"precision": "tf32 (split bf16 hi/lo operands, three tcgen05 MMAs per product)",
                                         "value": B / (ms3 / 1e3), "unit": "poses/s", "ms_per_step": ms3,
                                         "max_abs_err_over_scale": err3, "stated_bound": 1e-3}
            del m3

    if rank == 0:
        flops = spec.flops_per_pose(cfg)
        line = {
            "metric": metric_name(args), "value": value, "unit": "poses/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic",
            "config": {"workload": workload_name(args, cfg, B, f"batch {B} per GPU"), "arch": args.arch,
                       "batch_per_gpu": B, "views": cfg.V, "joints": cfg.J,
                       "parallelism": f"pose-sharded x{world}, no data-path collective",
                       "l2": "activation working set per step (GBs) far exceeds the 126 MB L2; no explicit flush",
                       "flops_per_pose": flops, "gemm_cta_group": int(os.environ.get("MPL_GEMM_CTA_GROUP", "0")) or None},
            "e2e": {"value": e2e_value, "unit": "poses/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": roofline, "whole_path_tflops": value / world * flops / 1e12,
            "breakdown": breakdown,
            "breakdown_note": "per-launch CUDA events on the launch stream in a separate profiled pass (same launches, same order as "
                              "the timed step); with chunk_streams=2 the timed step overlaps two chunks and runs below the sum",
            "breakdown_sum_ms": tot_ms / prof_steps, "memory_bound_kernels": memory_kernels, "hbm_peak_gbs": pk.get("hbm_gbs"),
            "cpu_baseline": cpu, "parity": parity, **extras, **({"dump_outputs": dump} if dump else {}),
            "mpjpe_cm": {"absolute": res["mpjpe_abs"], "root_relative": res["mpjpe_rel"], "procrustes_aligned": pres["p_mpjpe"],
                         "poses": res["n"],
                         "note": "random-init weights: the values only exercise the accumulators + all-reduce"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-gpu":
        run_reference_gpu(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
