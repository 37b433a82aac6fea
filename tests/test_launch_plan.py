"""The render launch policy (csrc/launch_plan.hpp) compiled into a small native harness: the automatic sample-range
schedules of the bench frame, the config-4 frames and a small frame stay what they were measured at, forced splits are
near-equal, every schedule covers the samples with non-empty ranges inside the 32-bit work counter, deep trees step
the CTA size down, and a row range maps to the tiles that cover it.  CPU only."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))


def test_launch_plan(tmp_path):
    exe = str(tmp_path / "launch_plan_check")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-o", exe, os.path.join(HERE, "native", "launch_plan_check.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count(" ok") == 6, r.stdout
