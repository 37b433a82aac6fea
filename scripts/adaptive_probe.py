#!/usr/bin/env python
"""Cost and benefit of tile-adaptive sampling (rt.render_adaptive) on one GPU; writes OUT/adaptive_probe.json.

For the bench frame (Weekend, 1200x800) and the earth frame (1920x1080):
  overhead  threshold 0 with max_samples 512 (every tile runs all passes) against a plain 512-spp render: the cost of
            the extra launches, merges and per-pass synchronisations alone; medians of 3 timed calls after a warm-up
  savings   thresholds of 2, 1 and 0.5 levels with max_samples 2048: mean spp, passes, kernel and total ms, Mrays/s, and
            the error against an 8192-spp reference of another seed (gamma space, in 8-bit levels: RMSE and 99th
            percentile), next to a uniform render with at least the same mean spp
and, for the 300x200 Weekend frame against the committed 4096-spp golden means (tests/golden/), the comparison
tests/test_adaptive.py makes, over a few thresholds, maximum counts and seeds.

    python scripts/adaptive_probe.py --out DIR
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import shirley_raytracing_rs_b200 as rt  # noqa: E402

LEVEL = 1.0 / 255.0


def gamma(x):
    return np.sqrt(np.clip(x, 0.0, 1.0))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError as e:
        q = f"nvidia-smi unavailable: {e}"
    return q


def passes_of(acc, initial):
    most, n, k = int(acc[..., 3].max()), initial, 1
    while n < most:
        n, k = n * 2, k + 1
    return k


def timed(fn, reps=3):
    fn()                                   # warm-up: module load, buffers
    runs = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        runs.append((time.perf_counter() - t0) * 1e3)
        st = out[-1]
    return out, st, float(np.median(runs))


def err_levels(img, ref):
    d = np.abs(img - ref) * 255.0
    return float(np.sqrt(np.mean(d ** 2))), float(np.quantile(d, 0.99))


def frame_probe(name, scene, cam):
    H, W = cam.image_height, cam.image_width
    res = {"frame": f"{W}x{H}"}
    (_, pst), _, p_wall = timed(lambda: rt.render(scene, cam, samples=512, seed=1))
    (_, _, ast), _, a_wall = timed(lambda: rt.render_adaptive(scene, cam, 512, 0.0, 16, seed=1))
    res["overhead_512spp"] = {
        "plain": {"kernel_ms": pst.kernel_ms, "total_ms": pst.total_ms, "wall_ms": p_wall, "launches": pst.launches, "rays": pst.rays},
        "adaptive_threshold0": {"kernel_ms": ast.kernel_ms, "total_ms": ast.total_ms, "wall_ms": a_wall, "launches": ast.launches, "rays": ast.rays,
                                "passes": len([16, 32, 64, 128, 256, 512])},
        "total_ms_ratio": ast.total_ms / pst.total_ms, "wall_ratio": a_wall / p_wall}
    ref_acc, _ = rt.render(scene, cam, samples=8192, seed=424242)
    ref = gamma(ref_acc[..., :3].astype(np.float64) / 8192)
    rows = []
    for levels in (2.0, 1.0, 0.5):
        (acc, _, st), _, wall = timed(lambda: rt.render_adaptive(scene, cam, 2048, levels * LEVEL, 16, seed=1), reps=1)
        mean_spp = st.paths / (W * H)
        e = err_levels(gamma(acc[..., :3].astype(np.float64) / acc[..., 3:4]), ref)
        spp = int(math.ceil(mean_spp))
        (uacc, ust), _, uwall = timed(lambda: rt.render(scene, cam, samples=spp, seed=1), reps=1)
        ue = err_levels(gamma(uacc[..., :3].astype(np.float64) / spp), ref)
        rows.append({"levels": levels, "max_samples": 2048, "initial_samples": 16,
                     "adaptive": {"mean_spp": mean_spp, "passes": passes_of(acc, 16), "kernel_ms": st.kernel_ms, "total_ms": st.total_ms,
                                  "wall_ms": wall, "mrays_per_s": st.rays / st.kernel_ms / 1e3, "rmse_levels": e[0], "p99_levels": e[1]},
                     "uniform": {"spp": spp, "kernel_ms": ust.kernel_ms, "total_ms": ust.total_ms, "wall_ms": uwall,
                                 "mrays_per_s": ust.rays / ust.kernel_ms / 1e3, "rmse_levels": ue[0], "p99_levels": ue[1]}})
        print(f"{name} {levels} levels: adaptive {mean_spp:.1f} spp rmse {e[0]:.3f} p99 {e[1]:.3f} {st.total_ms:.1f} ms | "
              f"uniform {spp} spp rmse {ue[0]:.3f} p99 {ue[1]:.3f} {ust.total_ms:.1f} ms", flush=True)
    res["savings_vs_8192spp_reference"] = rows
    return res


def block_stats(img, ref, b=10):
    H, W = ref.shape[:2]
    d = (img - ref)[: H - H % b, : W - W % b].reshape(H // b, b, W // b, b, -1)
    return np.sqrt((d ** 2).mean(axis=(1, 3, 4))).ravel(), d.mean(axis=(1, 3, 4)).ravel()


def golden_probe():
    """tests/test_adaptive.py's quality comparison over thresholds, maximum counts and seeds."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "weekend_mean_300x200_4096spp.npz"))
    ref = gamma(0.5 * (g["mean_a"].astype(np.float64) + g["mean_b"]))
    scene = rt.Scene.from_json(open(os.path.join(ROOT, "tests", "golden", "weekend_scene.json")).read(), 0x5EED)
    cam = rt.default_camera(300)
    worst = lambda r: float(np.sort(r)[-len(r) // 10:].mean())
    rows = []
    for max_samples in (256, 1024):
        for levels in (0.5, 1.0, 2.0, 4.0):
            for seed in (77, 78, 79):
                acc, _, st = rt.render_adaptive(scene, cam, max_samples, levels * LEVEL, 16, seed=seed)
                spp = int(math.ceil(st.paths / (cam.image_width * cam.image_height)))
                uni, _ = rt.render(scene, cam, samples=spp, seed=seed)
                a = gamma(acc[..., :3].astype(np.float64) / acc[..., 3:4])
                u = gamma(uni[..., :3].astype(np.float64) / spp)
                ra, ba = block_stats(a, ref)
                ru, bu = block_stats(u, ref)
                row = {"max_samples": max_samples, "levels": levels, "seed": seed, "mean_spp": st.paths / a[..., 0].size, "uniform_spp": spp,
                       "rmse": [float(np.sqrt(np.mean((a - ref) ** 2))), float(np.sqrt(np.mean((u - ref) ** 2)))],
                       "worst_decile_block_rmse": [worst(ra), worst(ru)],
                       "block_bias_max": [float(np.abs(ba).max()), float(np.abs(bu).max())],
                       "block_bias_rms": [float(np.sqrt(np.mean(ba ** 2))), float(np.sqrt(np.mean(bu ** 2)))]}
                rows.append(row)
                print("golden", json.dumps(row), flush=True)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    args = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("adaptive_probe needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    out = {"card": card(), "note": "times from CUDA events (kernel_ms: path-tracing kernels; total_ms: the whole call) and the host clock "
                                   "(wall_ms, includes the copy of the accumulation buffer to the host)"}
    out["golden_300x200"] = golden_probe()
    out["bench_1200x800"] = frame_probe("bench", rt.Scene.named("random", seed=0xDEADBEEF), rt.default_camera(1200))
    out["earth_1920x1080"] = frame_probe("earth", rt.Scene.named("earth"), rt.default_camera(1920, aspect_ratio=(16, 9)))
    with open(os.path.join(args.out, "adaptive_probe.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("card", "bench_1200x800", "earth_1920x1080")}, indent=1))


if __name__ == "__main__":
    main()
