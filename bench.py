#!/usr/bin/env python
"""bench.py — Mrays/s & ms/frame on the Weekend final scene, 1200x800, 500 spp, depth 50
(BASELINE.json metric; workload = configs[1]), on 1 / 2 / 4 / 8 B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE frame of the named workload: every pixel gets 500 samples of
ray_color(pixel_ray(..)) and the frame ends up as RGB8 on rank 0.  A "ray" is one closest-hit
query (one path segment, render.rs:31), counted by the kernel.

  value      whole-job Mrays/s with the scene resident in HBM, timed with CUDA events around each
             step on the launching stream (L2 flushed between steps), max over ranks.
  e2e        the same metric through the reference-facing call sequence with HOST (pageable)
             buffers: b200rt_scene_create (H2D of the flattened scene) + render + resolve + D2H
             of the RGB8 frame per step (N = 1: b200rt_render_rgb8).
  roofline   FP32-issue roofline of the path-tracing kernel (SURVEY.md §8d): algorithmic
             lane-ops per ray (24 per box test + 30 per primitive test + 70 fixed, from the
             kernel's own traversal counters) x rays / kernel time, against the FFMA-chain
             ceiling measured live on the same device.  The scene (~60 KB) lives in shared
             memory, so HBM is idle; its figures are added for completeness.
  cpu_baseline  the oracle (f64 restatement of the reference, OpenMP over scanlines = the
             reference's rayon row tasks) timed on this box's host cores on a bounded
             sample of the same frame (N = 1 only).
  other_configs  BASELINE configs 3-5, measured after the headline (outside its timed region):
             N = 1: C3 earth, C4 at 1e5 and 1e6 spheres; N > 1: C4 tile-sharded, C5 sample-sharded.

Multi-GPU (N > 1, one rank per GPU under torchrun) is STRONG scaling by default, like the
reference's parallel driver, which splits one frame over its workers (src/main.rs:92-126): the
500 samples of every pixel are split into N contiguous sample ranges (streams are keyed by
(pixel, sample), so the union is exactly the one-GPU frame); each rank renders its range into its
own float4 buffer and the buffers become one RGB8 frame on rank 0 inside the timed region — by
default with the fused peer-memory kernel (b200rt_resolve_peers_rgb8_device: every rank sums its
band of rows from all ranks' buffers over NVLink P2P, resolves and stores the bytes into rank 0's
frame; ranks ordered by flags in peer memory).  `--combine nccl` = NCCL reduce + resolve on rank 0.
Before the timed loop the N-rank frame is checked: byte-equal to gather + ordered sum +
resolve_kernel ("combine_check") and within one 8-bit level of the same frame rendered by rank 0
alone ("strong_check").  A flag wait that times out fails the run.
`--scaling weak` keeps round 1's measurement (every rank adds 500 samples of its own).

After the multi-process legs rank 0 alone renders the same strong-scaled frame over all N devices
through b200rt_multi_render_rgb8 — the single-process entry a Rust `render_scene` would call
(INTEGRATION.md §6) — reported as "e2e_single_process".

`--impl reference` times the reference's own CPU path (the oracle port — the Rust crate
cannot be built in this image) on the same config with all host threads.

`--dump-outputs DIR` writes what the last timed step computed, as float32 .npy files: at N = 1 the
accumulation buffer a caller of b200rt_render_device receives (DIR/accum.npy, [H, W, 4]: RGB sums and
the sample count), at N > 1 the RGB8 frame on rank 0 (DIR/frame.npy, [H, W, 3]).  Scene and seeds are
fixed, so two builds run with the same arguments can be compared output for output.  An output over
64 MiB is replaced by a fixed, seeded sample of its pixels, whose flat indices go to DIR/<name>_pixels.npy.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WIDTH, SPP, DEPTH, SCENE_SEED = 1200, 500, 50, 0xDEADBEEF
WORKLOAD = "weekend_final_scene_1200x800_500spp_depth50"
# ncu --set full of the C4 launches (scripts/profile_c4.py; profiles/r02_c4_metrics.md): bytes per 64-spp launch
C4_NCU = {"lts_1e6": 267870144256, "dram_1e6": 172336384, "lts_1e5": 178832932832, "dram_1e5": 110871296}
METRIC = "Mrays/s, Weekend final scene 1200x800 500spp (ms/frame in ms_per_step)"
DUMP_BYTES = 64 << 20          # --dump-outputs: at most this much per run


# stdout carries exactly ONE JSON line: anything else a library prints there (NCCL's version banner,
# for one) is redirected to stderr.
_JSON_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region.

    NVML is polled from a thread every 10 ms (the handle is opened in start(), before the timed region: an
    8-GPU strong-scaled run times 5 x 25 ms and a `nvidia-smi -lms` child has not printed its first line by then).
    Falls back to the `nvidia-smi -lms 100` loop of the profiling recipe when NVML cannot be opened."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index, uuid=None):
        self.index, self.uuid, self.proc, self.lines = index, uuid, None, []
        self.nvml, self.handle, self.samples, self.stop_flag, self.t = None, None, [], threading.Event(), None

    def _open_nvml(self):
        import pynvml
        pynvml.nvmlInit()
        h = None
        if self.uuid:
            for u in (f"GPU-{self.uuid}", str(self.uuid)):
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(u.encode() if isinstance(u, str) else u)
                    break
                except Exception:
                    h = None
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.nvml, self.handle = pynvml, h
        self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

    def _poll_nvml(self):
        n, h = self.nvml, self.handle
        while not self.stop_flag.is_set():
            try:
                sm = float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM))
                pw = n.nvmlDeviceGetPowerUsage(h) / 1000.0
                rs = int(n.nvmlDeviceGetCurrentClocksEventReasons(h))
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            self.stop_flag.wait(0.010)

    def start(self):
        try:
            self._open_nvml()
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self.stop_flag.set()
            self.t.join(timeout=2)
            n = self.nvml
            names = (("hw_slowdown", n.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", n.nvmlClocksEventReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", n.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", n.nvmlClocksEventReasonSwPowerCap))
            sm = sorted(s[0] for s in self.samples)
            reasons = sorted({name for s in self.samples for name, bit in names if s[2] & bit})
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.sm_max,
                    "power_w_max": max((s[1] for s in self.samples), default=None), "samples": len(sm), "reasons": reasons,
                    "source": "NVML polled every 10 ms during the timed steps"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons),
                "source": "nvidia-smi -lms 100 during the timed steps"}


def algorithmic_ops_per_ray(node_visits, prim_tests, rays):
    """SURVEY.md §8d: 24 lane-ops per box test (each node visit tests both children's boxes),
    30 per primitive test, 70 fixed per segment."""
    return 24.0 * (2.0 * node_visits / rays) + 30.0 * (prim_tests / rays) + 70.0


def algorithmic_bytes_per_ray(node_visits, prim_tests, rays):
    """64 B per node visit (one BVH2 node: both children's boxes + references), 16 B per primitive test
    (a sphere), 32 B of material per segment."""
    return 64.0 * (node_visits / rays) + 16.0 * (prim_tests / rays) + 32.0


def dump_output(out_dir, name, t, limit=DUMP_BYTES):
    """Writes tensor t ([H, W, C] on the device) as out_dir/<name>.npy in float32; over `limit` bytes, a fixed
    seeded sample of its pixels instead, with their flat indices in out_dir/<name>_pixels.npy (float64)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    a = t.float().cpu().numpy()
    if a.nbytes > limit:
        px = a.reshape(-1, a.shape[-1])
        n = (limit - 4096) // (px.shape[1] * 4 + 8)
        idx = np.sort(np.random.default_rng(0).choice(len(px), n, replace=False))
        np.save(os.path.join(out_dir, f"{name}_pixels.npy"), idx.astype(np.float64))
        a = px[idx]
    np.save(os.path.join(out_dir, f"{name}.npy"), a)
    log(f"dumped {name} {list(a.shape)} float32 to {out_dir}")


def workload_config(W, H, spp, world, scaling):
    name = WORKLOAD if (spp == SPP and W == WIDTH and scaling == "strong") else (
        f"weekend_{W}x{H}_{spp}spp_depth{DEPTH}" if scaling == "strong" else f"weekend_{W}x{H}_{spp * world}spp_depth{DEPTH}_weak_{spp}spp_per_gpu")
    return name


def run_reference(args, rank, world):
    """The reference arm: the oracle port on the host cores (rank 0 only)."""
    if rank != 0:
        return
    import shirley_raytracing_rs_b200 as rt
    from oracle import pyoracle as po
    scene = rt.Scene.named("random", seed=SCENE_SEED)
    cam = rt.default_camera(WIDTH)
    o = po.OracleScene(scene.desc, reference_topology=True, precision=64)
    cores = os.cpu_count() or 1
    spp = max(1, args.ref_spp)
    times, rays = [], 0
    for i in range(args.warmup + args.steps):
        _, st = o.render(cam, spp, max_depth=DEPTH, seed=1000 + i, threads=cores)
        if i >= args.warmup:
            times.append(st.seconds); rays += st.rays
    total = sum(times)
    val = rays / total / 1e6
    H = cam.image_height
    sample = f"{WIDTH}x{H} full frame at {spp} spp per step (of {SPP}), f64, OpenMP dynamic,1 over scanlines"
    d = scene.desc.contents
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Mrays/s", "n_gpus": 0, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / max(1, args.steps), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            # the same config keys as the b200 arm; the CPU arm renders a bounded sample of the frame per step and reports a RATE
            "config": {"workload": WORKLOAD, "scene": "src/scenes.rs random_scene (day), seeded", "scene_seed": SCENE_SEED, "objects": int(d.n_prims),
                       "image": [WIDTH, H], "spp": SPP, "max_depth": DEPTH, "parallelism": f"{cores} host threads over scanlines",
                       "normalised": f"rate over {spp} spp/step: a full {SPP}-spp CPU frame takes ~{1e3 * total / max(1, args.steps) * SPP / spp / 1e3:.0f} s, so each step renders {spp} of the {SPP} samples per pixel and Mrays/s is compared",
                       "sample": sample, "rays_per_step": rays // max(1, args.steps)},
            "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_JSON_OUT, flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--spp", type=int, default=SPP, help="samples per pixel of the frame (strong) or per GPU (weak); BASELINE: 500")
    ap.add_argument("--width", type=int, default=WIDTH)
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: split ONE spp-sample frame over the ranks (default; the BASELINE metric) or give every rank spp samples of its own")
    ap.add_argument("--ref-spp", type=int, default=16, help="spp of the bounded CPU sample per step")
    ap.add_argument("--cpu-baseline-spp", type=int, default=128, help="bounded CPU sample: ~10-30 s of host work")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true", help="skip BASELINE configs 3-5 after the headline")
    ap.add_argument("--no-single-process", action="store_true", help="N > 1: skip the b200rt_multi_render_rgb8 leg")
    ap.add_argument("--peer-barrier", default="flags", choices=["flags", "nccl"],
                    help="--combine peer: order the ranks with flags in peer memory (default) or a one-element NCCL all_reduce")
    ap.add_argument("--combine", default="peer", choices=["peer", "nccl"],
                    help="N > 1: fused peer-memory reduce+resolve kernel over NVLink (default) or NCCL reduce then resolve on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world != 1:
        log(f"warning: WORLD_SIZE={world} but --gpus {args.gpus}")

    import numpy as np
    import torch
    import torch.distributed as dist
    import shirley_raytracing_rs_b200 as rt
    from shirley_raytracing_rs_b200 import sharding
    F, lib = rt._ffi, rt._ffi.lib

    if not torch.cuda.is_available() or rt.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    ctl = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        ctl = dist.new_group(backend="gloo")      # host-side barriers that leave the GPUs idle (the single-process leg)

    scene = rt.Scene.named("random", seed=SCENE_SEED)
    cam = rt.default_camera(args.width)
    W, H = cam.image_width, cam.image_height
    dscene = scene.device(local_rank)
    info = scene.info(local_rank)
    stream = torch.cuda.current_stream()
    sptr = C.c_void_p(stream.cuda_stream)
    strong = args.scaling == "strong" or world == 1
    total_spp = args.spp if strong else args.spp * world
    my = sharding.sample_ranges(total_spp, world)[rank] if strong else sharding.weak_sample_range(args.spp, rank)
    if my.samples == 0:
        raise SystemExit(f"--spp {args.spp} leaves rank {rank} of {world} without samples")
    peer = None
    if world > 1 and args.combine == "peer":
        peer = sharding.PeerFrame(W, H, local_rank, barrier=args.peer_barrier)   # IPC-shared accumulation buffers, flags, the frame on rank 0
        accum = peer.accum()
    else:
        accum = torch.zeros((H, W, 4), dtype=torch.float32, device=dev)
    frame_dev = torch.empty((H, W, 3), dtype=torch.uint8, device=dev) if (world > 1 and peer is None and rank == 0) else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def params(step, count=False, rng=my):
        return F.RenderParams(samples=rng.samples, sample_offset=rng.sample_offset, max_depth=DEPTH,
                              flags=F.FLAG_COUNT_TRAVERSAL if count else 0, seed=77 + step, device=-1)

    def combine():
        """N > 1: the per-rank buffers become ONE RGB8 frame on rank 0 (stream-ordered; rank 0's stream ends after the last band landed)."""
        if peer is not None:
            peer.combine(total_spp, sptr)             # barrier, fused sum+resolve of this rank's row band into rank 0's frame, "done" signal
            if rank == 0:
                peer.wait_frame(sptr)                 # every rank's band is in the frame
        else:
            dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)
            if rank == 0:
                F.check(lib.b200rt_resolve_rgb8_device(accum.data_ptr(), W, H, total_spp, frame_dev.data_ptr(), sptr))

    def frame(step, count=False, handle=dscene):
        """One step with the scene resident in HBM: render (+ at N > 1 the cross-GPU sum and resolve)."""
        p = params(step, count)
        if peer is not None:
            peer.begin_frame(sptr)
        F.check(lib.b200rt_render_device(handle, C.byref(cam), C.byref(p), accum.data_ptr(), sptr))
        if world > 1:
            combine()

    def finish(handle=dscene):
        st = F.Stats()
        F.check(lib.b200rt_render_device_finish(handle, sptr, C.byref(st)))
        if peer is not None:
            peer.check()                              # a flag wait that gave up on a peer fails the run
        return st

    def frame_on_rank0():
        return peer.frame_tensor() if peer is not None else frame_dev

    # ---- counters run (untimed): traversal statistics for the roofline -----------------------
    frame(0, count=True)
    cst = finish()
    cnt = torch.tensor([float(cst.node_visits), float(cst.prim_tests), float(cst.rays), float(cst.paths)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    c_nodes, c_prims, c_rays, c_paths = [float(x) for x in cnt.tolist()]
    ops_per_ray = algorithmic_ops_per_ray(c_nodes, c_prims, c_rays)
    bytes_per_ray = algorithmic_bytes_per_ray(c_nodes, c_prims, c_rays)

    # ---- N > 1 correctness, where the driver sees it -------------------------------------------
    checks = {}
    if world > 1:
        frame(1); finish()
        torch.cuda.synchronize()
        gathered = [torch.empty_like(accum) for _ in range(world)] if rank == 0 else None
        dist.gather(accum.contiguous(), gathered, dst=0)
        if rank == 0:
            got = frame_on_rank0().clone()
            tot = gathered[0].clone()
            for r in range(1, world):
                tot += gathered[r]                     # the fused kernel's order: rank 0, 1, 2, ...
            want = torch.empty((H, W, 3), dtype=torch.uint8, device=dev)
            F.check(lib.b200rt_resolve_rgb8_device(tot.data_ptr(), W, H, total_spp, want.data_ptr(), sptr))
            torch.cuda.synchronize()
            if peer is not None:
                if not torch.equal(got, want):
                    raise SystemExit("combine_check FAILED: fused peer-memory resolve differs from gather + ordered sum + resolve_kernel")
                checks["combine_check"] = "ok"
            else:
                d = (got.int() - want.int()).abs()
                if int(d.max()) > 1:
                    raise SystemExit("combine_check FAILED: NCCL reduce + resolve differs from the ordered sum by more than one level")
                checks["combine_check"] = f"ok (NCCL sum order: max diff {int(d.max())} level)"
            if strong:
                # the same frame rendered by this GPU alone: all samples, same seed
                solo = torch.empty((H, W, 4), dtype=torch.float32, device=dev)
                p = params(1, rng=sharding.SampleRange(0, total_spp))
                F.check(lib.b200rt_render_device(dscene, C.byref(cam), C.byref(p), solo.data_ptr(), sptr))
                st1 = F.Stats(); F.check(lib.b200rt_render_device_finish(dscene, sptr, C.byref(st1)))
                F.check(lib.b200rt_resolve_rgb8_device(solo.data_ptr(), W, H, total_spp, want.data_ptr(), sptr))
                torch.cuda.synchronize()
                d = (got.int() - want.int()).abs()
                if int(d.max()) > 1:
                    raise SystemExit(f"strong_check FAILED: the {world}-GPU frame differs from the 1-GPU frame by {int(d.max())} levels")
                checks["strong_check"] = {"max_level_diff": int(d.max()), "pixels_differing": float((d > 0).any(dim=-1).float().mean()),
                                          "one_gpu_ms": st1.kernel_ms, "note": "N-rank frame vs the same 500-spp frame on rank 0 alone (f32 partial sums: +-1 level)"}
        dist.barrier()

    # ---- warm-up ---------------------------------------------------------------------------------
    for i in range(args.warmup):
        frame(i); finish()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    fp32_peak = rt.fp32_peak(local_rank)   # lane-instr/s, measured live (FFMA chain)

    # ---- timed steps -----------------------------------------------------------------------------
    sampler = ClockSampler(local_rank, getattr(torch.cuda.get_device_properties(local_rank), "uuid", None))
    sampler.start()
    step_ms, kernel_ms, rays, launches = [], [], 0, 0
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)                       # L2 flush between timed iterations
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        frame(100 + i)
        e1.record(stream)
        st = finish()
        e1.synchronize()
        step_ms.append(e0.elapsed_time(e1)); kernel_ms.append(st.kernel_ms)
        rays += st.rays; launches += st.launches
        if world > 1:
            # peer: resolve_peers_kernel + the flag kernels (begin-frame wait, signal, wait, signal; + the frame wait on rank 0);
            # nccl: resolve_kernel on rank 0
            launches += ((5 if args.peer_barrier == "flags" else 1) + (1 if rank == 0 and args.peer_barrier == "flags" else 0)) if peer is not None else (1 if rank == 0 else 0)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    total_ms = float(sum(step_ms))
    if args.dump_outputs:
        # before the e2e leg, which renders into the same buffers at N > 1
        if world == 1:
            dump_output(args.dump_outputs, "accum", accum)
        elif rank == 0:
            dump_output(args.dump_outputs, "frame", frame_on_rank0())
        if world > 1:
            dist.barrier()

    # ---- e2e: the reference-facing call with host buffers -----------------------------------------
    rgb = np.empty((H, W, 3), dtype=np.uint8)                      # pageable, like a Rust Vec<u8>
    rgb_t = torch.from_numpy(rgb)
    e2e_ms, e2e_rays = [], 0
    h2d = int(info.device_bytes)
    d2h = H * W * 3

    def e2e_step(step):
        """scene upload + render + resolve + D2H of the frame, like render_scene (main.rs:65-130)."""
        t0 = time.perf_counter()
        h = C.c_void_p()
        F.check(lib.b200rt_scene_create(scene.desc, local_rank, C.byref(h)))
        try:
            st = F.Stats()
            if world == 1:
                p = params(step)
                F.check(lib.b200rt_render_rgb8(h, C.byref(cam), C.byref(p), rgb.ctypes.data, None, C.byref(st)))
            else:
                frame(step, handle=h)
                st = finish(handle=h)
                if rank == 0:
                    rgb_t.copy_(frame_on_rank0())
                torch.cuda.synchronize()
        finally:
            lib.b200rt_scene_destroy(h)
        ms = (time.perf_counter() - t0) * 1e3
        log(f"[rank {rank}] e2e step {step}: {ms:.2f} ms wall (kernel {st.kernel_ms:.2f} ms, device total {st.total_ms:.2f} ms)")
        return ms, st.rays

    e2e_step(0)
    if world > 1:
        dist.barrier()
    for i in range(args.steps):
        ms, r = e2e_step(200 + i)
        e2e_ms.append(ms); e2e_rays += r
    if world > 1:
        dist.barrier()

    # ---- per-frame fixed cost, itemised with CUDA events (one extra frame, untimed otherwise) -----------------------
    breakdown = None
    if world > 1 and peer is not None and args.peer_barrier == "flags":
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
        torch.cuda.synchronize(); dist.barrier()
        ev[0].record(stream)
        peer.begin_frame(sptr)
        ev[1].record(stream)
        p = params(300)
        F.check(lib.b200rt_render_device(dscene, C.byref(cam), C.byref(p), accum.data_ptr(), sptr))
        ev[2].record(stream)
        peer.combine(total_spp, sptr, events=(lambda k: ev[3 + k].record(stream)))   # after signal+wait, after resolve, after the done signal
        if rank == 0:
            peer.wait_frame(sptr)
        ev[6].record(stream)
        bst = finish()
        torch.cuda.synchronize()
        names = ["begin_frame_wait", "render (memset counters + kernel)", "ready signal + wait for all ranks", "fused sum+resolve of this rank's band",
                 "done signal", "wait for all bands (rank 0)"]
        mine = [ev[k].elapsed_time(ev[k + 1]) for k in range(6)]
        t = torch.tensor(mine + [bst.kernel_ms], dtype=torch.float64, device=dev)
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tmin = t.clone(); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        if rank == 0:
            breakdown = {"unit": "ms, one frame, CUDA events on each rank's stream: [rank 0, min over ranks, max over ranks]",
                         **{n: [round(mine[k], 4), round(float(tmin[k]), 4), round(float(tmax[k]), 4)] for k, n in enumerate(names)},
                         "path_trace_kernel_v2": [round(bst.kernel_ms, 4), round(float(tmin[6]), 4), round(float(tmax[6]), 4)]}
        dist.barrier()

    # ---- reduce over ranks: max time, sum rays ----------------------------------------------------
    vals = torch.tensor([total_ms, float(sum(e2e_ms)), float(sum(kernel_ms))], dtype=torch.float64, device=dev)
    cnts = torch.tensor([float(rays), float(e2e_rays), float(launches)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnts, op=dist.ReduceOp.SUM)
    total_ms, e2e_total_ms, kernel_total_ms = [float(x) for x in vals.tolist()]
    rays_all, e2e_rays_all, launches_all = [float(x) for x in cnts.tolist()]

    # ---- single-process leg: rank 0 alone drives all N devices through b200rt_multi_render_rgb8 -------------------
    single = None
    if world > 1 and strong and not args.no_single_process:
        torch.cuda.synchronize()
        dist.barrier(group=ctl)
        if rank == 0:
            try:
                devs = (C.c_int * world)(*range(world))
                mh = C.c_void_p()
                F.check(lib.b200rt_multi_create(devs, world, C.byref(mh)))
                sp_ms, sp_rays = [], 0
                for i in range(args.warmup + args.steps):
                    p = F.RenderParams(samples=total_spp, max_depth=DEPTH, seed=400 + i, device=-1)
                    st = F.Stats()
                    t0 = time.perf_counter()
                    F.check(lib.b200rt_multi_render_rgb8(mh, scene.desc, C.byref(cam), C.byref(p), rgb.ctypes.data, C.byref(st)))
                    ms = (time.perf_counter() - t0) * 1e3
                    if i >= args.warmup:
                        sp_ms.append(ms); sp_rays += st.rays
                    log(f"[single-process x{world}] frame {i}: {ms:.2f} ms wall (slowest kernel {st.kernel_ms:.2f} ms)")
                lib.b200rt_multi_destroy(mh)
                single = {"value": sp_rays / (sum(sp_ms) * 1e-3) / 1e6, "unit": "Mrays/s", "ms_per_step": sum(sp_ms) / len(sp_ms),
                          "path": f"b200rt_multi_render_rgb8 over devices 0..{world - 1} from ONE host process: scene upload per device, sample ranges, "
                                  "fused peer-access sum+resolve on device 0, RGB8 into a pageable host buffer",
                          "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h}
            except F.B200rtError as e:
                single = {"error": str(e)}
        dist.barrier(group=ctl)

    # ---- BASELINE configs 3-5 (outside the headline's timed region) ------------------------------------------------
    other = None
    if not args.no_other_configs:
        try:
            other = other_configs(rt, sharding, rank, world, local_rank, dev, stream, sptr, fp32_peak)
        except Exception as e:       # the headline stands on its own
            other = {"error": f"{type(e).__name__}: {e}"}
            log(f"[rank {rank}] other_configs failed: {e}")

    if rank == 0:
        value = rays_all / (total_ms * 1e-3) / 1e6
        e2e_value = e2e_rays_all / (e2e_total_ms * 1e-3) / 1e6
        k_rays_per_s = (rays / len(kernel_ms)) / (np.mean(kernel_ms) * 1e-3)     # this rank's kernel alone
        achieved = k_rays_per_s * ops_per_ray                                      # lane-ops/s
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        roofline = {"bound": "fp32-issue", "achieved": achieved / 1e12, "peak": fp32_peak / 1e12, "unit": "Tlane-op/s",
                    "frac": achieved / fp32_peak if fp32_peak else None,
                    # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel (ncu --set full,
                    # profiles/): the scene is staged in shared memory, HBM is idle
                    "traffic": 23805200, "traffic_unit": "bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum of one 500-spp launch (ncu --set full, profiles/r02_ncu_metrics.md, last column): 23.18 MB read + 0.63 MB written; the 15 MB accumulation buffer and the 23 MB fixed-point sums of the chunked tiles stay in L2",
                    "kernel": "path_trace_kernel_v2", "kernel_ms": float(np.mean(kernel_ms)),
                    "ops_per_ray": ops_per_ray, "node_visits_per_ray": c_nodes / c_rays, "prim_tests_per_ray": c_prims / c_rays,
                    "segments_per_sample": c_rays / c_paths,
                    "peak_source": "FFMA-chain microbenchmark run live in this process (b200rt_fp32_peak); MEASURED_PEAKS.json has no FP32 figure",
                    "hbm": {"bound": "hbm", "achieved": k_rays_per_s * bytes_per_ray / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": k_rays_per_s * bytes_per_ray / 1e9 / hbm_peak, "bytes_per_ray": bytes_per_ray,
                            "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                            "note": "algorithmic bytes are served from shared memory (scene staged per CTA), not HBM"}}
        if world == 1:
            par, e2e_path = "single GPU", "b200rt_scene_create + b200rt_render_rgb8 (pageable host RGB8 out) per step"
        else:
            how = "fused peer-memory sum+resolve (NVLink P2P)" if peer is not None else "NCCL reduce + resolve on rank 0"
            par = (f"ONE {total_spp}-spp frame split into {world} sample ranges of {total_spp // world}-{-(-total_spp // world)} spp, " if strong
                   else f"weak: {args.spp} spp per GPU, {total_spp} spp frame, sample-range x{world}, ") + how
            e2e_path = ("per rank and step: b200rt_scene_create + b200rt_render_device on the rank's sample range + combine ("
                        + ("b200rt_peer_signal/wait_device + b200rt_resolve_peers_rgb8_device" if peer is not None else "NCCL reduce + b200rt_resolve_rgb8_device")
                        + ") + b200rt_render_device_finish; rank 0 copies the RGB8 frame into a pageable host buffer")
        line = {"metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": workload_config(W, H, args.spp, world, "strong" if strong else "weak"),
                           "scene": "src/scenes.rs random_scene (day), seeded", "scene_seed": SCENE_SEED, "objects": int(info.n_prims),
                           "bvh_nodes": int(info.n_bvh_nodes), "image": [W, H], "spp": total_spp, "spp_per_gpu": total_spp / world, "max_depth": DEPTH,
                           "parallelism": par,
                           "l2": "256 MiB buffer written between timed steps (outside the per-step CUDA events)",
                           "rays_per_step": rays_all / args.steps, "Msamples_per_s": (W * H * total_spp) / (total_ms / args.steps * 1e-3) / 1e6},
                "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": h2d * world, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_total_ms / args.steps,
                        "path": e2e_path, "host_buffer": "pageable"},
                "gpu_launches": int(launches_all),
                "clocks": clocks, "roofline": roofline, "wall_s": wall}
        line.update(checks)
        if breakdown is not None:
            line["frame_breakdown"] = breakdown
        if single is not None:
            line["e2e_single_process"] = single
        if other is not None:
            line["other_configs"] = other
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as po
            o = po.OracleScene(scene.desc, reference_topology=True, precision=64)
            cores = os.cpu_count() or 1
            o.render(cam, 1, max_depth=DEPTH, seed=5, threads=cores)     # warm
            _, ost = o.render(cam, args.cpu_baseline_spp, max_depth=DEPTH, seed=6, threads=cores)
            _, o1 = o.render(cam, 2, max_depth=DEPTH, seed=7, threads=1)   # the reference's --single-threaded twin (src/main.rs:97-112), 2 spp
            line["cpu_baseline"] = {"value": ost.rays / ost.seconds / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
                                    "single_thread_value": o1.rays / o1.seconds / 1e6,
                                    "sample": f"{W}x{H} full frame at {args.cpu_baseline_spp} spp (of {args.spp}), f64 oracle, OpenMP dynamic,1 over scanlines, {ost.seconds:.1f} s",
                                    "pops_per_ray": ost.pops / ost.rays, "leaf_tests_per_ray": ost.leaf_tests / ost.rays}
        print(json.dumps(line), file=_JSON_OUT, flush=True)
    if peer is not None:
        peer.close()
    if world > 1:
        dist.destroy_process_group()


def other_configs(rt, sharding, rank, world, local_rank, dev, stream, sptr, fp32_peak):
    """BASELINE configs 3-5 on this many GPUs, one timed frame each (after a warm-up frame), CUDA events, max over ranks.
    N = 1: C3 (earth, the real assets/earthmap.jpg), C4 at 1e5 and 1e6 spheres.  N > 1: C4 (1e6 spheres) tile-sharded, C5
    (Weekend 3840x2160, 4096 spp) sample-sharded through the fused peer-memory resolve."""
    import numpy as np
    import torch
    import torch.distributed as dist
    F, lib = rt._ffi, rt._ffi.lib
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    l2_peak = rt.read_peak(48 << 20, local_rank)          # GB/s, float4 loads over a 48 MiB (L2-resident) buffer, measured live

    def run(name, scene, cam, total_spp, mode):
        W, H = cam.image_width, cam.image_height
        h = scene.device(local_rank)
        info = scene.info(local_rank)
        pf = sharding.PeerFrame(W, H, local_rank) if world > 1 else None
        accum = pf.accum() if pf is not None else torch.empty((H, W, 4), dtype=torch.float32, device=dev)
        rgb = torch.empty((H, W, 3), dtype=torch.uint8, device=dev) if pf is None else None
        if mode == "tiles":
            sc, si = sharding.tile_shard(world, rank)
            base = dict(samples=total_spp, sample_offset=0, shard_count=sc, shard_index=si)
        else:
            sr = sharding.sample_ranges(total_spp, world)[rank]
            base = dict(samples=sr.samples, sample_offset=sr.sample_offset)

        def one(seed, count):
            p = F.RenderParams(max_depth=DEPTH, seed=seed, device=-1, flags=F.FLAG_COUNT_TRAVERSAL if count else 0, **base)
            if pf is not None:
                pf.begin_frame(sptr)
            F.check(lib.b200rt_render_device(h, C.byref(cam), C.byref(p), accum.data_ptr(), sptr))
            if pf is not None:
                pf.combine(total_spp, sptr)
                if rank == 0:
                    pf.wait_frame(sptr)
            else:
                F.check(lib.b200rt_resolve_rgb8_device(accum.data_ptr(), W, H, total_spp, rgb.data_ptr(), sptr))
            st = F.Stats()
            F.check(lib.b200rt_render_device_finish(h, sptr, C.byref(st)))
            if pf is not None:
                pf.check()
            return st

        # warm-up + traversal counters: the same frame once, untimed (first use of a frame size allocates the library's
        # per-stream scratch — counters, the fixed-point sums of chunked tiles — which must not land in the timed frame)
        cst = one(1, True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = one(2, False)
        e1.record(stream); e1.synchronize()
        t = torch.tensor([e0.elapsed_time(e1), st.kernel_ms], dtype=torch.float64, device=dev)
        r = torch.tensor([float(st.rays), float(st.paths), float(cst.rays), float(cst.node_visits), float(cst.prim_tests)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX); dist.all_reduce(r, op=dist.ReduceOp.SUM)
        ms, kms = float(t[0]), float(t[1])
        rays, paths, crays, cnodes, cprims = [float(x) for x in r.tolist()]
        out = None
        if rank == 0:
            opr = algorithmic_ops_per_ray(cnodes, cprims, crays)
            bpr = algorithmic_bytes_per_ray(cnodes, cprims, crays)
            rps = rays / (ms * 1e-3)
            in_smem = int(info.bvh_nodes_in_smem) == int(info.n_bvh_nodes)
            out = {"workload": name, "n_gpus": world, "sharding": mode if world > 1 else "single GPU", "image": [W, H], "spp": total_spp, "objects": int(info.n_prims),
                   "bvh_nodes": int(info.n_bvh_nodes), "bvh_depth": int(info.bvh_depth), "bvh_builder": "device LBVH" if info.bvh_builder else "host SAH",
                   "scene_device_bytes": int(info.device_bytes), "scene_in_shared_memory": in_smem,
                   "value": rps / 1e6, "unit": "Mrays/s", "ms_per_frame": ms, "kernel_ms_max": kms, "Msamples_per_s": paths / (ms * 1e-3) / 1e6,
                   "segments_per_sample": rays / paths, "node_visits_per_ray": cnodes / crays, "prim_tests_per_ray": cprims / crays,
                   "roofline": {"bound": "fp32-issue", "achieved": rps * opr / 1e12, "peak": fp32_peak * world / 1e12, "unit": "Tlane-op/s",
                                "frac": rps * opr / (fp32_peak * world), "ops_per_ray": opr}}
            if not in_smem:
                # The tree lives in global memory and is served mostly by L1 and L2 (ncu, profiles/r02_c4_metrics.md: L1 hit rate
                # ~80-91 %, L2 ~83-88 %): algorithmic node + primitive bytes per ray x rays/s against the L2 read ceiling measured
                # live (b200rt_read_peak over 48 MiB) and against the HBM figure of MEASURED_PEAKS.json.  `traffic` = what one
                # 64-spp launch of this kernel moved at L2 (lts__t_bytes.sum) and at DRAM (dram__bytes_read + write), from ncu.
                ncu = {"c4_1e6": {"lts_bytes": C4_NCU.get("lts_1e6"), "dram_bytes": C4_NCU.get("dram_1e6")}, "c4_1e5": {"lts_bytes": C4_NCU.get("lts_1e5"), "dram_bytes": C4_NCU.get("dram_1e5")}}
                key = "c4_1e6" if info.n_prims > 500000 else "c4_1e5"
                out["roofline_bytes"] = {"bound": "l2", "achieved": rps * bpr / 1e9, "peak": l2_peak * world, "unit": "GB/s", "frac": rps * bpr / 1e9 / (l2_peak * world),
                                         "bytes_per_ray": bpr, "peak_source": "b200rt_read_peak(48 MiB) measured live (L2-resident float4 reads)",
                                         "hbm": {"peak": hbm_peak * world, "frac": rps * bpr / 1e9 / (hbm_peak * world), "peak_source": "MEASURED_PEAKS.json hbm_gbs"},
                                         "traffic": ncu[key]["dram_bytes"], "traffic_l2": ncu[key]["lts_bytes"],
                                         "traffic_unit": "bytes per 64-spp single-GPU launch (ncu --set full, profiles/r02_c4_metrics.md): dram__bytes_read.sum + dram__bytes_write.sum; traffic_l2 = lts__t_bytes.sum",
                                         "note": "algorithmic bytes (64 B per node visit, 16 B per primitive test, 32 B material per ray) are mostly L1 hits; L2 and DRAM see the miss traffic"}
        if pf is not None:
            pf.close()
        scene.close()
        return out

    res = {}
    if world == 1:
        res["c3_earth_1920x1080_256spp"] = run("C3 textured earth sphere (assets/earthmap.jpg), 1920x1080, 256 spp", rt.Scene.named("earth"),
                                               rt.default_camera(1920, aspect_ratio=(16, 9)), 256, "samples")
        for G, tag in ((158, "c4_1e5_3840x2160_64spp"), (500, "c4_1e6_3840x2160_64spp")):
            camG = rt.camera((0.9 * G, 0.18 * G + 2, 0.35 * G), (0, 0, 0), vfov=30, aperture=0.001, width=3840, aspect_ratio=(16, 9), focus_length=10.0)
            res[tag] = run(f"C4 scaled random spheres G={G}, 3840x2160, 64 spp", rt.Scene.named("scaled", seed=3, param=G), camG, 64, "samples")
    else:
        G = 500
        camG = rt.camera((0.9 * G, 0.18 * G + 2, 0.35 * G), (0, 0, 0), vfov=30, aperture=0.001, width=3840, aspect_ratio=(16, 9), focus_length=10.0)
        res["c4_1e6_3840x2160_64spp_tiles"] = run(f"C4 scaled random spheres G={G}, 3840x2160, 64 spp, interleaved tile shards", rt.Scene.named("scaled", seed=3, param=G), camG, 64, "tiles")
        res["c5_weekend_3840x2160_4096spp"] = run("C5 Weekend final scene 3840x2160, 4096 spp, sample ranges + fused peer-memory resolve",
                                                  rt.Scene.named("random", seed=SCENE_SEED), rt.default_camera(3840, aspect_ratio=(16, 9)), 4096, "samples")
    return res if rank == 0 else None


if __name__ == "__main__":
    main()
