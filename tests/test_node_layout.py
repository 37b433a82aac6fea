"""The BVH node packing (csrc/node_layout.hpp) compiled into a small native harness: over random, degenerate, empty and
non-finite child boxes, each child's centre/half-extent box read back from the child-paired slots contains the builder's
box, the node carries both child references, and the node is the previous child-major layout with its slots permuted.
CPU only."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))


def test_node_layout(tmp_path):
    exe = str(tmp_path / "node_layout_check")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-o", exe, os.path.join(HERE, "native", "node_layout_check.cpp")])
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[:3] == ["contain ok", "refs ok", "permuted ok"], r.stdout
