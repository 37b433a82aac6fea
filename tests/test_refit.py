"""The BVH refit of b200rt_scene_update through its host twin (csrc/prim_box.hpp), compiled into a small native harness with
g++: over host SAH trees of random and degenerate primitives (coincident, thin, huge, inverted, NaN) and a hand-built
Karras-numbered tree, the links name every parent and leaf slot, a refit from unchanged records reproduces the builder's
nodes byte for byte, and after random moves every child box is the packed exact union of its subtree's padded leaf boxes.
CPU only."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))


def test_refit(tmp_path):
    exe = str(tmp_path / "refit_check")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-fopenmp", "-o", exe, os.path.join(HERE, "native", "refit_check.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[:4] == ["links ok", "noop ok", "moved ok", "karras ok"], r.stdout
