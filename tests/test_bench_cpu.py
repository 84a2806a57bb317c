"""bench.py: argument checks, the --dump-outputs writer, the step count of the reference arm, and (GPU) that the dump is
the output of the timed path."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench


def _run_bench(*argv):
    r = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), *argv], capture_output=True, text=True,
                       timeout=600, env=dict(os.environ, OMP_NUM_THREADS="2"))
    assert r.returncode == 0, r.stderr[-2000:]
    return json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])


def _parse(monkeypatch, *argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    return bench.parse()


def test_steps_and_dump_outputs_arguments(monkeypatch):
    a = _parse(monkeypatch, "--steps", "7", "--dump-outputs", "d")
    assert a.steps == 7 and a.dump_outputs == "d"
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]):
        with pytest.raises(SystemExit):
            _parse(monkeypatch, *argv)


def test_dump_outputs_writes_the_step_output_whole_or_a_fixed_sample(tmp_path, monkeypatch):
    out = torch.arange(50 * 17 * 3, dtype=torch.float32).reshape(50, 17, 3)
    info = bench.dump_outputs(str(tmp_path / "a"), out)
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "output.npy"), out.numpy())
    assert info["shape"] == [50, 17, 3] and info["sample"] is None
    monkeypatch.setattr(bench, "DUMP_LIMIT", 10 * 17 * 3 * 4)          # room for 10 poses
    for d in ("b", "c"):
        info = bench.dump_outputs(str(tmp_path / d), out)
    b, c = np.load(tmp_path / "b" / "output.npy"), np.load(tmp_path / "c" / "output.npy")
    assert b.shape == (10, 17, 3) and b.dtype == np.float32 and info["poses_of"] == 50
    np.testing.assert_array_equal(b, c)                                  # same poses on every run
    rows = b[:, 0, 0] / (17 * 3)
    assert np.all(np.diff(rows) > 0) and np.array_equal(b, out.numpy()[rows.astype(int)])


def test_reference_arm_times_exactly_the_requested_steps():
    d = _run_bench("--impl", "reference", "--steps", "101", "--warmup", "1", "--depth", "1", "--cpu-batch", "4")
    assert d["steps"] == 101 and d["cpu_baseline"]["sample"].startswith("101 forwards")


@pytest.mark.gpu
def test_dump_is_the_output_of_the_last_timed_step(tmp_path, monkeypatch):
    """The dumped array equals a direct forward of the same seeded weights and inputs through the module."""
    from openmpl_b200 import spec, synth
    from openmpl_b200.models.multiview_mpl_b200 import MultiView_MPL
    argv = ["--batch", "1000", "--depth", "2", "--steps", "2", "--warmup", "1"]
    d = _run_bench(*argv, "--no-cpu-baseline", "--no-extras", "--parity-poses", "0", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2 and d["dump_outputs"]["ranks"] == [0] and d["dump_outputs"]["sample"] is None
    kw, cfg = bench.workload(_parse(monkeypatch, *argv))
    m = MultiView_MPL(**kw, precision="bf16")
    m.load_state_dict({k: torch.from_numpy(v) for k, v in synth.named_weights(spec.param_spec(cfg), seed=0).items()})
    m = m.cuda().eval()
    batch = synth.make_batch(1000, synth.make_rig(cfg.V, bench.ARCH_RIG["hm0"]), seed=1, start=0)
    x = {k: torch.from_numpy(batch[k]).cuda() for k in ("poses", "rays", "centers")}
    with torch.no_grad():
        out = m(x["poses"], rays=x["rays"], centers=x["centers"])
    np.testing.assert_array_equal(np.load(tmp_path / "output.npy"), out.cpu().numpy())
