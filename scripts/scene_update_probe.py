#!/usr/bin/env python
"""Cost of b200rt_scene_update against b200rt_scene_create, and the tree-quality drift of a refit BVH; writes
OUT/scene_update_probe.json (default OUT: profiles/).

create vs update   for the Weekend scene (485 objects, host SAH), `scaled` G=158 (~1e5 spheres, host SAH) and G=500 (~1e6,
                   device LBVH): host wall time of scene_create and of scene_update for a moved description (medians of 5).
                   Device side, from the library's B200RT_TIMING report: for create, the synchronous upload ("cudaMalloc +
                   H2D") and the tree build (B200rtSceneInfo.bvh_build_ms: CUDA events for the device LBVH, host time for
                   the host SAH build); for update, the CUDA events recorded around its copies and the refit kernel
                   ("H2D + refit (device)", "refit kernel (device)"), and the first update's link derivation
drift              every sphere but the up-front primitives moves along its own direction by a fixed step per frame; after
                   k = 1, 10 and 60 frames of updates, rays/s (median of 3 renders without counters) and BVH node visits per
                   ray (one counting render) of the refit tree against a tree built from the same description

    python scripts/scene_update_probe.py [--out DIR]
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import shirley_raytracing_rs_b200 as rt  # noqa: E402

F = rt._ffi


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError as e:
        return f"nvidia-smi unavailable: {e}"


class Dev:
    def __init__(self, desc):
        self.h = C.c_void_p()
        F.check(F.lib.b200rt_scene_create(desc, 0, C.byref(self.h)))

    def device(self, device=-1):
        return self.h

    def info(self):
        out = F.SceneInfo()
        F.check(F.lib.b200rt_scene_info(self.h, C.byref(out)))
        return out

    def close(self):
        F.lib.b200rt_scene_destroy(self.h)


def spheres(scene):
    d = scene.desc.contents
    return np.ctypeslib.as_array(C.cast(d.spheres, C.POINTER(C.c_float)), shape=(d.n_spheres, 4))


def median_ms(fn, n):
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def timing_report(fn):
    """Runs fn with B200RT_TIMING=1 and returns the library's phase report from stderr: {(call, phase): ms}."""
    os.environ["B200RT_TIMING"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["B200RT_TIMING"]
        tmp.seek(0)
        text = tmp.read()
    out = {}
    for m in re.finditer(r"\[b200rt\] (scene_\w+) (.+?)\s+([0-9.]+) ms", text):
        out[(m.group(1), m.group(2).strip())] = out.get((m.group(1), m.group(2).strip()), 0.0) + float(m.group(3))
    return out


CONFIGS = [
    ("weekend", lambda: rt.Scene.named("random", seed=0xDEADBEEF), lambda: rt.default_camera(640), 16),
    ("scaled_158", lambda: rt.Scene.named("scaled", seed=11, param=158),
     lambda: rt.camera((142, 30.4, 55.3), (0, 0, 0), vfov=30, aperture=0.001, width=640, aspect_ratio=(16, 9), focus_length=10.0), 4),
    ("scaled_500", lambda: rt.Scene.named("scaled", seed=11, param=500),
     lambda: rt.camera((450, 92, 175), (0, 0, 0), vfov=30, aperture=0.001, width=640, aspect_ratio=(16, 9), focus_length=10.0), 4),
]
STEP = 0.05          # scene units per frame (neighbouring spheres of these scenes are about one unit apart)


def probe(name, make, make_cam, spp):
    s = make()
    base = spheres(s).copy()
    rng = np.random.default_rng(1)
    ang = rng.uniform(0, 2 * np.pi, len(base))
    vel = np.stack([np.cos(ang), np.zeros_like(ang), np.sin(ang)], axis=1).astype(np.float32) * STEP
    movable = base[:, 3] < 50.0
    vel[~movable] = 0

    def frame(k):
        spheres(s)[:, :3] = base[:, :3] + k * vel

    r = {"n_prims": int(s.desc.contents.n_prims)}
    devs = []
    r["create_host_ms"] = median_ms(lambda: devs.append(Dev(s.desc)), 5)
    for d in devs[1:]:
        d.close()
    dev = devs[0]
    info = dev.info()
    r["builder"] = "lbvh" if info.bvh_builder else "sah"
    r["create_bvh_build_ms"] = float(info.bvh_build_ms)
    r["n_bvh_nodes"] = int(info.n_bvh_nodes)
    rep = timing_report(lambda: Dev(s.desc).close())
    r["create_upload_ms"] = rep.get(("scene_create", "cudaMalloc + H2D"), float("nan"))
    frame(1)
    rep = timing_report(lambda: F.check(F.lib.b200rt_scene_update(dev.h, s.desc)))   # the first update also derives the links
    r["first_update_links_ms"] = rep.get(("scene_update", "refit links (first update)"), float("nan"))
    ks = iter(range(2, 100))
    r["update_host_ms"] = median_ms(lambda: (frame(next(ks)), F.check(F.lib.b200rt_scene_update(dev.h, s.desc))), 5)
    reps = [timing_report(lambda: (frame(next(ks)), F.check(F.lib.b200rt_scene_update(dev.h, s.desc)))) for _ in range(5)]
    r["update_device_ms"] = float(np.median([x[("scene_update", "H2D + refit (device)")] for x in reps]))
    r["refit_kernel_ms"] = float(np.median([x[("scene_update", "refit kernel (device)")] for x in reps]))

    cam = make_cam()
    drift = []
    dev.close()
    frame(0)                                 # drift: a tree built at frame 0, then k frames of motion
    dev = Dev(s.desc)
    k_done = 0
    for k in (1, 10, 60):
        for j in range(k_done + 1, k + 1):   # every frame is one update, as a host animating the scene would do
            frame(j)
            F.check(F.lib.b200rt_scene_update(dev.h, s.desc))
        k_done = k
        fresh = Dev(s.desc)
        row = {"k": k}
        for label, h in (("refit", dev), ("rebuilt", fresh)):
            rt.render(h, cam, samples=spp, seed=1)
            rates = []
            for _ in range(3):
                _, st = rt.render(h, cam, samples=spp, seed=1)
                rates.append(st.rays / st.kernel_ms / 1e3)
            _, stc = rt.render(h, cam, samples=spp, seed=1, count_traversal=True)
            row[label] = {"mrays_per_s": float(np.median(rates)), "node_visits_per_ray": stc.node_visits / stc.rays}
        fresh.close()
        row["visits_ratio"] = row["refit"]["node_visits_per_ray"] / row["rebuilt"]["node_visits_per_ray"]
        row["rate_ratio"] = row["refit"]["mrays_per_s"] / row["rebuilt"]["mrays_per_s"]
        drift.append(row)
        print(name, row, flush=True)
    r["drift"] = drift
    dev.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    if rt.device_count() < 1:
        raise SystemExit("scene_update_probe needs a CUDA device")
    out = {"card": card(), "step_per_frame": STEP, "configs": {}}
    for name, make, make_cam, spp in CONFIGS:
        if args.only and name not in args.only.split(","):
            continue
        out["configs"][name] = probe(name, make, make_cam, spp)
        out["configs"][name]["spp"] = spp
        print(name, {k: v for k, v in out["configs"][name].items() if k != "drift"}, flush=True)
    out["card_after"] = card()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "scene_update_probe.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
