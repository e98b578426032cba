"""bench.py contract on a CPU box: the reference arm (the oracle timed as the reference's CPU implementation) prints
ONE JSON line with the keys the driver reads; the product arm refuses to run without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["metric"] == "frames/sec @368x368 2-scale" and d["value"] > 0 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return  # the -m gpu suite and the driver exercise the product arm on a GPU box
    r = _run("--steps", "1", "--warmup", "0")
    assert r.returncode != 0  # no CPU fallback: the product path fails loudly
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same arrays, bit for bit, and they are the joints of
    the bench frames (every step feeds the same frames, so the filtered joints stay those of one estimate).  --steps
    sets the number of timed steps: the kernel launches counted inside the timed loop scale with it."""
    from oracle import synth
    from vnect_b200 import VNectEngine
    from vnect_b200.weights import seeded_init
    nf = 4
    dumps, lines = [], []
    for run, steps in (("a", 3), ("b", 3), ("c", 6)):
        d = tmp_path / run
        r = _run("--steps", str(steps), "--warmup", "0", "--frames", str(nf), "--no-cpu-baseline", "--no-c4",
                 "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-3000:]
        out = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        assert len(out) == 1
        lines.append(json.loads(out[0]))
        assert lines[-1]["steps"] == steps
        assert sorted(os.listdir(d)) == ["joints_2d.npy", "joints_3d.npy"]
        dumps.append((np.load(d / "joints_2d.npy"), np.load(d / "joints_3d.npy")))
    launches = [ln["gpu_launches"] for ln in lines]
    assert launches[0] > 0 and launches[1] == launches[0] and launches[2] == 2 * launches[0], launches
    (a2, a3), (b2, b3), _ = dumps
    assert a2.dtype == np.float64 and a2.shape == (nf, 21, 2)
    assert a3.dtype == np.float32 and a3.shape == (nf, 21, 3)
    assert np.array_equal(a2, b2) and np.array_equal(a3, b3)
    eng = VNectEngine(seeded_init("W0"), [1.0, 0.7], max_frames=nf, max_streams=nf)
    try:
        j2, j3 = eng.estimate(np.stack([synth.frame_c2(i) for i in range(nf)]), np.arange(nf), 1.0, 1.004)
    finally:
        eng.close()
    assert np.abs(a2 - j2).max() < 1e-6 and np.abs(a3.astype(np.float64) - j3).max() < 1e-2
