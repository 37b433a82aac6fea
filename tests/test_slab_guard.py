"""The fast-slab guard (csrc/launch_plan.hpp: fast_slab_ok) compiled into a small native harness with the centre-form slab
test restated lane by lane in fmaf: on boxes padded and packed as scene creation does it, whenever the guard allows the fast
form and a ray meets the unpadded box (f64), the fast form enters the box — at scales 1e-3 to 1e6, origins up to the guard's
limit, directions down to its limit and components that are 0, subnormal or below the 1e-18 reciprocal clamp.  The pinned
case is a short ray (|d| = 1e-15) that the fast form would cull.  CPU only."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))


def test_slab_guard(tmp_path):
    exe = str(tmp_path / "slab_guard_check")
    # -ffp-contract=off: the harness's plain a * b must not be fused, its fmaf stand for the device's FFMA2 lanes
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-ffp-contract=off", "-o", exe,
                           os.path.join(HERE, "native", "slab_guard_check.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[:3] == ["pinned ok", "sweep ok", "needed ok"], r.stdout
