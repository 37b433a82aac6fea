"""Tile-adaptive sampling's arithmetic (csrc/adaptive_plan.hpp) compiled into a small native harness: the pass schedule, the
per-pixel error estimate against a float64 numpy restatement of the formula in include/b200rt.h, and the size of the ABI struct.
CPU only."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ONE = 2.0 ** 32          # the fixed-point scale of the per-pixel sums


def error_f64(n, s, F, P):
    """e_p per row, in float64; also the bound of the f32 rounding of the two means the kernel takes."""
    n, s = n[:, None].astype(np.float64), s[:, None].astype(np.float64)
    a = np.minimum(F / ONE / n, 1.0)
    b = np.minimum(P / ONE / s, 1.0)
    m = np.minimum((F + P) / ONE / (n + s), 1.0)
    k = np.sqrt(n * s) / (n + s)
    scale = k / (2.0 * np.sqrt(np.maximum(m, 2.0 ** -16)))
    e = (np.abs(a - b) * scale).max(axis=1)
    rounding = (np.maximum(np.abs(a), np.abs(b)) * scale).max(axis=1) * 8 * 2.0 ** -24
    return e, rounding


def cases():
    rng = np.random.default_rng(20261020)
    rows = []
    # random scenes of the usual brightness: per-sample radiance mostly below 1, sums of n and s samples
    for _ in range(4000):
        n = int(rng.choice([1, 2, 16, 32, 64, 256, 1024]))
        s = int(rng.choice([1, n, max(1, n // 3)]))
        mu = rng.uniform(0, 1.2, 3)
        F = np.round(rng.gamma(2.0, mu / 2.0 + 1e-9, 3) * n * ONE)
        P = np.round(rng.gamma(2.0, mu / 2.0 + 1e-9, 3) * s * ONE)
        rows.append((n, s, *F, *P))
    rows += [(16, 16, 0, 0, 0, 0, 0, 0),                         # black: no error
             (1, 1, 0, 0, 0, 1, 1, 1),                           # one fixed-point unit: below the 2^-16 floor of m
             (16, 16, 16 * ONE, 20 * ONE, 40 * ONE, 16 * ONE, 30 * ONE, 17 * ONE),   # saturated in both means: 0
             (16, 16, 8 * ONE, 8 * ONE, 8 * ONE, 24 * ONE, 8 * ONE, 8 * ONE),        # one mean saturated
             (32, 32, 2 ** 61, 2 ** 60, 3 * 2 ** 59, 5, 7, 11),   # emitter-bright sums near the 63-bit limit against a dark pass
             (2048, 2048, 2 ** 62, 2 ** 62, 2 ** 62, 2 ** 62 - 2 ** 40, 2 ** 40, 0),
             (1, 2 ** 20, 3 * ONE, 0, ONE // 2, ONE, 2 ** 20 * ONE // 4, 7 * ONE)]
    return np.array(rows, dtype=np.float64)


def test_adaptive_plan(tmp_path, rt):
    exe = str(tmp_path / "adaptive_plan_check")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-o", exe, os.path.join(HERE, "native", "adaptive_plan_check.cpp")])
    x = cases()
    stdin = "\n".join(" ".join(str(int(v)) for v in row) for row in x) + "\n"
    r = subprocess.run([exe], input=stdin, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == "schedule ok", r.stdout
    assert lines[1] == f"sizeof {C.sizeof(rt._ffi.AdaptiveParams)}" == "sizeof 16"
    got = np.array([float(v) for v in lines[2:]])
    assert got.shape == (len(x),)
    want, rounding = error_f64(x[:, 0], x[:, 1], x[:, 2:5], x[:, 5:8])
    assert np.all(np.abs(got - want) <= 1e-5 * want + rounding), np.max(np.abs(got - want) - 1e-5 * want - rounding)
    assert got[-7] == 0.0 and got[-5] == 0.0
    assert got[-6] > 0.0 and got[-4] > 0.0 and got[-3] > 0.0
    assert np.all(np.isfinite(got)) and (got[:-7] > 0).mean() > 0.9
