"""The denoiser's arithmetic (csrc/denoise_plan.hpp) compiled into a small native harness: the edge-stopping weight and the
two-halves variance against a float64 numpy restatement of the formulas in the header, on random, zero-variance, miss and
degenerate-albedo inputs, plus the tap tables and the size of the ABI struct.  CPU only."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SIGMA_L, EPS_L, SIGMA_N, SIGMA_Z, SIGMA_A = 4.0, 1e-10, 128.0, 0.05, 0.1


def weight_f64(x):
    lp, lq, vbar = x[:, 0], x[:, 1], x[:, 2]
    np_, zp, nq, zq = x[:, 3:6], x[:, 6], x[:, 7:10], x[:, 10]
    ap, aq, dist = x[:, 11:14], x[:, 14:17], x[:, 17]
    wl = np.exp(-np.abs(lp - lq) / (SIGMA_L * np.sqrt(np.maximum(vbar, 0.0)) + EPS_L))
    nn = np.sqrt((np_ ** 2).sum(1) * (nq ** 2).sum(1))
    c = np.where(nn > 0, np.minimum((np_ * nq).sum(1) / np.where(nn > 0, nn, 1.0), 1.0), 0.0)
    wn = np.where(c > 0, np.maximum(c, 0.0) ** SIGMA_N, 0.0)
    zm = np.maximum(zp, zq)
    wz = np.where(zm > 0, np.exp(-np.abs(zp - zq) / (SIGMA_Z * np.where(zm > 0, zm, 1.0) * dist)), 1.0)
    wa = np.exp(-np.abs(ap - aq).sum(1) / SIGMA_A)
    w = wl * wn * wz * wa
    return np.where((zp == 0) != (zq == 0), 0.0, w)


def variance_f64(x):
    la, lb, na, nb = x[:, 18], x[:, 19], x[:, 20], x[:, 21]
    ok = (na > 0) & (nb > 0)
    return np.where(ok, (la - lb) ** 2 * na * nb / np.where(ok, na + nb, 1.0) ** 2, 0.0)


def cases():
    rng = np.random.default_rng(20261021)
    n = 3000
    x = np.zeros((n, 22))
    x[:, 0:2] = rng.uniform(0, 2, (n, 2))
    x[:, 2] = rng.choice([0.0, 1e-4, 1e-2, 0.3], n)                     # zero variance included
    nrm = rng.normal(size=(n, 2, 3))
    nrm /= np.linalg.norm(nrm, axis=2, keepdims=True)
    near = rng.random(n) < 0.5                                          # many nearly parallel normals: wn far from 0
    nrm[near, 1] = nrm[near, 0] + 0.05 * rng.normal(size=(near.sum(), 3))
    x[:, 3:6], x[:, 7:10] = nrm[:, 0], nrm[:, 1]
    x[:, 6] = rng.uniform(0.5, 20, n)
    x[:, 10] = x[:, 6] * rng.uniform(0.9, 1.1, n)
    miss = rng.random(n)
    x[miss < 0.1, 6] = 0.0                                             # p missed
    x[miss < 0.1, 3:6] = 0.0
    x[(miss >= 0.1) & (miss < 0.2), 10] = 0.0                          # q missed
    x[(miss >= 0.1) & (miss < 0.2), 7:10] = 0.0
    both = (miss >= 0.2) & (miss < 0.25)
    x[both, 6] = x[both, 10] = 0.0
    x[:, 11:14] = rng.uniform(0, 1, (n, 3))
    x[:, 14:17] = np.clip(x[:, 11:14] + 0.05 * rng.normal(size=(n, 3)), 0, 1)
    x[rng.random(n) < 0.05, 14:17] = 0.0                                # black albedo
    x[:, 17] = rng.choice([1, 2, 4, 8, 16, 32], n)
    x[:, 18:20] = rng.uniform(0, 3, (n, 2))
    x[:, 20] = rng.choice([0, 1, 2, 8, 512], n)
    x[:, 21] = rng.choice([1, 2, 9, 512], n)
    x[:20, 18] = x[:20, 19]                                             # equal halves: no variance
    return x.astype(np.float32).astype(np.float64)


def test_denoise_plan(tmp_path, rt):
    exe = str(tmp_path / "denoise_plan_check")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-o", exe, os.path.join(HERE, "native", "denoise_plan_check.cpp")])
    x = cases()
    stdin = "\n".join(" ".join(repr(float(v)) for v in row) for row in x) + "\n"
    r = subprocess.run([exe], input=stdin, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == f"sizeof {C.sizeof(rt._ffi.DenoiseParams)}" == "sizeof 16"
    assert lines[1] == "taps 1 1"
    got = np.array([[float(v) for v in ln.split()] for ln in lines[2:]])
    assert got.shape == (len(x), 2)
    w, v = weight_f64(x), variance_f64(x)
    # f32 evaluation: exp of arguments up to ~1e3 in magnitude and a 128th power carry ~1e-4 relative rounding
    assert np.all(np.abs(got[:, 0] - w) <= 2e-4 * w + 1e-30), np.max(np.abs(got[:, 0] - w) / np.maximum(w, 1e-30))
    assert np.all(np.abs(got[:, 1] - v) <= 1e-5 * v + 1e-30)
    assert np.all(got >= 0) and np.all(np.isfinite(got))
    mixed = (x[:, 6] == 0) != (x[:, 10] == 0)
    assert mixed.sum() > 100 and np.all(got[mixed, 0] == 0.0)          # sky never mixes with geometry
    assert (got[~mixed & (x[:, 6] > 0), 0] > 1e-3).mean() > 0.2        # and the random cases do exercise non-zero weights
    assert np.all(got[:20, 1] == 0.0) and np.all(got[x[:, 20] == 0, 1] == 0.0)
