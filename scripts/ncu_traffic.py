#!/usr/bin/env python
"""Regenerate profiles/ncu_traffic.json (what bench.py reports as roofline.traffic) from an `ncu --set full` capture of the
four FPT GEMM launches of one block, stamped with the build it was taken from.

    python scripts/ncu_traffic.py gpurun_out/<capture>.ncu-rep [arch] [profiles/<summary>.md] [gpurun_out/<head capture>.ncu-rep]

The optional fourth argument is a capture of head_block_kernel: its DRAM bytes per launch are recorded next to the GEMMs'
(reading the pose half of interleaved [x_j | ray_j] rows fetched whole 128-byte lines, twice the algorithmic bytes; the
channel-permuted residual planes made the half rows contiguous).
"""
import csv
import hashlib
import io
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"4": "qkv_ln_bias", "5": "fc1_ln_bias_gelu", "6": "proj_residual_emit", "7": "fc2_residual_emit"}


def main():
    rep = sys.argv[1]
    arch = sys.argv[2] if len(sys.argv) > 2 else "hm0"
    src = sys.argv[3] if len(sys.argv) > 3 else rep
    out = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(out)))
    hdr, units = rows[0], rows[1]
    ix = {h: i for i, h in enumerate(hdr)}

    def val(r, k):
        v, u = float(r[ix[k]].replace(",", "")), units[ix[k]].lower()
        return v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(u, 1)
    per, tens = {}, {}
    for r in rows[2:]:
        name = r[ix["Kernel Name"]]
        if "qkv_attn_kernel" in name:
            key = "qkv_attention_fused"
        elif "gemm_tcgen05_kernel" in name:
            epi = name.split("gemm_tcgen05_kernel<")[1].split(">")[0].replace("(int)", "").split(",")[-1].strip()
            key = NAMES.get(epi, "epi" + epi)
        else:
            continue
        n = 2
        while key in per:                      # two launches of one instantiation (D = 544: proj and fc2 share an epilogue)
            key = key.split("#")[0] + f"#{n}"
            n += 1
        per[key] = (val(r, "dram__bytes_read.sum") + val(r, "dram__bytes_write.sum")) / 1e6
        tens[key] = float(r[ix["sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"]])
    lib = os.path.join(ROOT, "openmpl_b200", "libmpl_b200.so")
    rev = subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], capture_output=True, text=True).stdout.strip()
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        data = json.load(open(path))
    except Exception:
        data = {}
    data[arch] = {"gemm_tcgen05_kernel": {
        "bytes_per_launch": 1e6 * sum(per.values()) / max(len(per), 1),
        "note": "mean over the FPT GEMM instantiations of one block (" + ", ".join(f"{k} {v:.0f} MB" for k, v in per.items())
                + f"), ncu --set full, chunk of 32768 poses, {os.path.basename(src)}",
        "per_instantiation_mb": per, "tensor_pipe_pct_ncu": tens,
        "capture": os.path.basename(rep), "git_rev_at_capture": rev,
        "lib_sha256_16": hashlib.sha256(open(lib, "rb").read()).hexdigest()[:16] if os.path.isfile(lib) else None}}
    if len(sys.argv) > 4:
        out2 = subprocess.run(["ncu", "-i", sys.argv[4], "--page", "raw", "--csv"], capture_output=True, text=True).stdout
        rows2 = list(csv.reader(io.StringIO(out2)))
        ix2 = {h: i for i, h in enumerate(rows2[0])}

        def val2(r, k):
            v, u = float(r[ix2[k]].replace(",", "")), rows2[1][ix2[k]].lower()
            return v * {"byte": 1, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9, "ns": 1e-9, "us": 1e-6, "usecond": 1e-6, "nsecond": 1e-9, "ms": 1e-3, "msecond": 1e-3}.get(u, 1)
        heads = [r for r in rows2[2:] if "head_block_kernel" in r[ix2["Kernel Name"]]]
        if heads:
            b = sum(val2(r, "dram__bytes_read.sum") + val2(r, "dram__bytes_write.sum") for r in heads) / len(heads)
            t = sum(val2(r, "gpu__time_duration.sum") for r in heads) / len(heads)
            data[arch]["head_block_kernel"] = {"bytes_per_launch": b, "ncu_launch_s": t, "ncu_dram_gbs": b / t / 1e9,
                                               "capture": os.path.basename(sys.argv[4]),
                                               "note": "DRAM bytes of one head launch (32768 poses), ncu --set full.  Channel-permuted "
                                                       "residual planes: contiguous half rows, traffic = algorithmic bytes; with the "
                                                       "reference's interleaved [x_j | ray_j] order it read whole 128-byte lines (2x)"}
    json.dump(data, open(path, "w"), indent=1)
    print(json.dumps(data[arch], indent=1))


if __name__ == "__main__":
    main()
