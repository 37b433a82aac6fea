#!/usr/bin/env python
"""Cost and benefit of the feature-guided à-trous denoiser (rt.render_denoised) on one GPU; writes OUT/denoise_probe.json.

overhead     device time of the feature pass at k = 1 and 4 feature rays per pixel and of one filter iteration, from
             torch.profiler's CUDA kernel records (medians of 3 calls after a warm-up), on the bench frame (Weekend, 1200x800)
             and the earth frame (1920x1080), next to the path-tracing kernel time of 4 spp of the same frame
equal time   gamma-space RMSE of the denoised n-spp frame against a noisy frame with n' spp, n' chosen so that its
             path-tracing time matches the denoised frame's device time (render + features + filter), for n = 8, 16, 64, on
             the 300x200 Weekend frame against the committed 4096-spp golden means and on the 150x150 Cornell box against a
             4096-spp render of another seed
quality      the ratios tests/test_denoise.py checks (16 and 1024 spp), at three seeds

    python scripts/denoise_probe.py --out DIR
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import shirley_raytracing_rs_b200 as rt  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def gamma(x):
    return np.sqrt(np.clip(x, 0.0, 1.0))


def rmse(x, ref):
    return float(np.sqrt(np.mean((x - ref) ** 2)))


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError as e:
        return f"nvidia-smi unavailable: {e}"


def kernel_ms(fn):
    """Device time per kernel-name group of one call of fn, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    groups = {"features": 0.0, "filter_iteration": 0.0, "demodulate": 0.0, "path_trace": 0.0, "iterations": 0}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        if "denoise_feature_kernel" in ev.name:
            groups["features"] += us / 1e3
        elif "denoise_atrous_kernel" in ev.name:
            groups["filter_iteration"] += us / 1e3
            groups["iterations"] += 1
        elif "denoise_demodulate_kernel" in ev.name:
            groups["demodulate"] += us / 1e3
        elif "path_trace_kernel_v2" in ev.name:
            groups["path_trace"] += us / 1e3
    return groups


def median_groups(fn, reps=3):
    fn()
    runs = [kernel_ms(fn) for _ in range(reps)]
    return {k: float(np.median([r[k] for r in runs])) for k in runs[0]}


def overhead(scene, cam):
    out = {}
    for k in (1, 4):
        g = median_groups(lambda: rt.render_denoised(scene, cam, 4, feature_samples=k, iterations=5))
        out[f"features_k{k}_ms"] = g["features"]
        out["filter_per_iteration_ms"] = g["filter_iteration"] / max(g["iterations"], 1)
        out["demodulate_ms"] = g["demodulate"]
        out["path_trace_4spp_ms"] = g["path_trace"]
    out["features_k4_plus_5_iterations_over_4spp"] = (out["features_k4_ms"] + out["demodulate_ms"] + 5 * out["filter_per_iteration_ms"]) / out["path_trace_4spp_ms"]
    return out


def equal_time(scene, cam, ref, seed):
    rows = []
    for n in (8, 16, 64):
        g = median_groups(lambda: rt.render_denoised(scene, cam, n, seed=seed))
        t_dn = g["path_trace"] + g["features"] + g["demodulate"] + g["filter_iteration"]
        per_spp = g["path_trace"] / n
        n_eq = max(n, int(round(t_dn / per_spp)))
        den, acc, _, _ = rt.render_denoised(scene, cam, n, seed=seed)
        noisy, _ = rt.render(scene, cam, samples=n_eq, seed=seed)
        rows.append({"n": n, "denoised_device_ms": t_dn, "noisy_spp_at_equal_time": n_eq,
                     "rmse_denoised": rmse(gamma(den[..., :3] / den[..., 3:]), ref),
                     "rmse_noisy_n": rmse(gamma(acc[..., :3] / n), ref),
                     "rmse_noisy_equal_time": rmse(gamma(noisy[..., :3] / n_eq), ref)})
        print(rows[-1], flush=True)
    return rows


def cornell(width):
    return rt.Scene.named("cornell"), rt.camera((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), vfov=40.0, focal_length=1.0,
                                                aperture=0.00001, width=width, aspect_ratio=(1, 1), focus_length=10.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="output directory")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    out = {"card": card()}
    out["bench_1200x800"] = overhead(rt.Scene.named("random", seed=0xDEADBEEF), rt.default_camera(1200))
    out["earth_1920x1080"] = overhead(rt.Scene.named("earth"), rt.default_camera(1920, aspect_ratio=(16, 9)))
    print(json.dumps(out, indent=1), flush=True)

    g = np.load(os.path.join(GOLDEN, "weekend_mean_300x200_4096spp.npz"))
    wref = gamma(0.5 * (g["mean_a"].astype(np.float64) + g["mean_b"]))
    wscene = rt.Scene.from_json(open(os.path.join(GOLDEN, "weekend_scene.json")).read(), 0x5EED)
    wcam = rt.default_camera(300)
    cscene, ccam = cornell(150)
    cacc, _ = rt.render(cscene, ccam, samples=4096, seed=102)
    cref = gamma(cacc[..., :3].astype(np.float64) / 4096)
    out["equal_time_weekend_300x200"] = equal_time(wscene, wcam, wref, 101)
    out["equal_time_cornell_150x150"] = equal_time(cscene, ccam, cref, 101)
    quality = []
    for seed in (101, 202, 303):
        for name, scene, cam, ref in (("weekend", wscene, wcam, wref), ("cornell", cscene, ccam, cref)):
            for n in (16, 1024):
                den, acc, _, _ = rt.render_denoised(scene, cam, n, seed=seed)
                rd, rn = rmse(gamma(den[..., :3] / den[..., 3:]), ref), rmse(gamma(acc[..., :3] / n), ref)
                quality.append({"scene": name, "seed": seed, "n": n, "rmse_denoised": rd, "rmse_noisy": rn, "ratio": rd / rn})
                print(quality[-1], flush=True)
    out["quality_ratios"] = quality
    with open(os.path.join(args.out, "denoise_probe.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
