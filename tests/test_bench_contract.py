"""bench.py's output contract, on the arm that runs without a GPU: `--impl reference` times the reference's CPU
path (the oracle port, the one other place bench.py may execute oracle/) and prints exactly ONE JSON line.
On the GPU: what `--dump-outputs` writes is what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-spp", "1", "--gpus", "1"],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"].startswith("Mrays/s") and d["config"]["workload"] == "weekend_final_scene_1200x800_500spp_depth50"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 1 and d["warmup"] == 0 and d["dtype"] == "f64"


@pytest.mark.gpu
@pytest.mark.parametrize("width,sampled", [(120, False), (2600, True)])    # 2600x1733 float4 is over the 64 MiB budget
def test_dump_outputs_is_the_last_timed_step(tmp_path, rt, gpu_required, width, sampled):
    """--dump-outputs writes the accumulation buffer of the last of --steps timed steps (seed 77 + 100 + steps - 1);
    an output over the budget becomes a seeded sample of its pixels."""
    steps, spp, out = 2, 3, tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--spp", str(spp),
                        "--width", str(width), "--no-cpu-baseline", "--no-other-configs", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    cam = rt.default_camera(width)
    want, _ = rt.render(rt.Scene.named("random", seed=0xDEADBEEF), cam, samples=spp, max_depth=50, seed=77 + 100 + steps - 1)
    got = np.load(out / "accum.npy")
    assert got.dtype == np.float32
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    if sampled:
        idx = np.load(out / "accum_pixels.npy")
        assert idx.dtype == np.float64 and np.all(np.diff(idx) > 0) and got.shape == (len(idx), 4) and len(idx) > 1_000_000
        want = want.reshape(-1, 4)[idx.astype(np.int64)]
    assert np.array_equal(got, want)


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"],
                       capture_output=True, text=True, cwd=ROOT, env=env, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""
