"""Tile-adaptive sampling (b200rt_render_adaptive, rt.render_adaptive, ray-cli --adaptive).

The per-pixel sums are exact 64-bit integers, so a tile that stopped after n samples must equal a plain n-sample render of
it bit for bit, and the stopping decisions can be recomputed from plain renders.  Renders are bit-deterministic: none of
these checks is statistical except the quality comparison, which runs at a fixed seed."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "ray-cli")
LEVEL = 1.0 / 255.0


def schedule(initial, max_samples):
    """n_0, n_1, ... up to max_samples (include/b200rt.h)."""
    n = [min(initial, max_samples)]
    while n[-1] < max_samples:
        n.append(min(n[-1] * 2, max_samples))
    return n


def tile_view(a, H, W):
    """[H, W, ...] -> [ceil(H/4), ceil(W/8), 32, ...], padded with NaN: the 8x4 tiles of the adaptive grid."""
    ty, tx = (H + 3) // 4, (W + 7) // 8
    pad = np.full((ty * 4, tx * 8) + a.shape[2:], np.nan, dtype=np.float64)
    pad[:H, :W] = a
    return pad.reshape(ty, 4, tx, 8, *a.shape[2:]).swapaxes(1, 2).reshape(ty, tx, 32, *a.shape[2:])


def tile_counts(acc, rows):
    """The one sample count of every tile's selected pixels (-1: none selected)."""
    H, W = acc.shape[:2]
    w = acc[..., 3].astype(np.float64)
    sel = np.zeros((H, W), bool)
    sel[rows[0]:rows[1]] = True
    w[~sel] = np.nan
    t = tile_view(w, H, W)
    hi, lo = np.where(np.isnan(t), -np.inf, t).max(axis=2), np.where(np.isnan(t), np.inf, t).min(axis=2)
    assert np.array_equal(hi[np.isfinite(hi)], lo[np.isfinite(lo)]), "a tile's pixels have different sample counts"
    return np.where(np.isfinite(hi), hi, -1).astype(np.int64)


@pytest.mark.gpu
def test_tiles_equal_plain_renders_bit_for_bit(rt, weekend, gpu_required):
    cam = rt.default_camera(150)                   # 150 x 100: a ragged last tile column
    rows = (5, 97)                                 # neither end on a tile boundary
    H, W = cam.image_height, cam.image_width
    acc, err, st = rt.render_adaptive(weekend, cam, max_samples=64, threshold=1.5 * LEVEL, initial_samples=4, seed=3,
                                      sample_offset=7, rows=rows)
    counts = tile_counts(acc, rows)
    assert err.shape == counts.shape == (25, 19)
    assert np.all(err[0] == -1) and np.all(err[1:] >= 0) and np.all(counts[0] == -1)
    assert np.all(acc[: rows[0]] == 0) and np.all(acc[rows[1]:] == 0)
    used = sorted(set(counts[counts > 0].tolist()))
    assert len(used) >= 2 and set(used) <= set(schedule(4, 64)[1:]), used
    for n in used:
        plain, _ = rt.render(weekend, cam, samples=n, seed=3, sample_offset=7, rows=rows)
        mine = np.repeat(np.repeat(counts == n, 4, axis=0), 8, axis=1)[:H, :W]
        assert np.array_equal(acc[mine], plain[mine]), n
    assert st.paths == int(acc[..., 3].sum())


@pytest.mark.gpu
def test_extremes(rt, weekend, gpu_required):
    cam = rt.default_camera(96)
    acc, err, _ = rt.render_adaptive(weekend, cam, max_samples=48, threshold=0.0, initial_samples=5, seed=11)
    plain, _ = rt.render(weekend, cam, samples=48, seed=11)
    assert np.array_equal(acc, plain)                      # threshold 0: every tile runs to max_samples
    assert np.all(err >= 0)
    for initial, max_samples in ((5, 48), (40, 64)):
        acc, _, _ = rt.render_adaptive(weekend, cam, max_samples=max_samples, threshold=1e30, initial_samples=initial, seed=11)
        assert np.all(acc[..., 3] == min(2 * initial, max_samples))   # nothing stops before its first estimate


def expected_tile_errors(rt, scene, cam, initial, max_samples, seed):
    """e_T of every tile after every pass k >= 1, from plain renders of [0, n_{k-1}), [n_{k-1}, n_k) and [0, n_k), in float64.
    The kernel reads the same float32 values: (float)sum * 2^-32 of the same integer sums."""
    H, W = cam.image_height, cam.image_width
    n = schedule(initial, max_samples)
    total = {m: rt.render(scene, cam, samples=m, seed=seed)[0].astype(np.float64) for m in n}
    out = []
    for k in range(1, len(n)):
        a_n, s = n[k - 1], n[k] - n[k - 1]
        part = rt.render(scene, cam, samples=s, seed=seed, sample_offset=a_n)[0].astype(np.float64)
        a = np.minimum(total[a_n][..., :3] / a_n, 1.0)
        b = np.minimum(part[..., :3] / s, 1.0)
        m = np.minimum(total[n[k]][..., :3] / n[k], 1.0)
        e = (np.abs(a - b) * np.sqrt(a_n * s) / (a_n + s) / (2 * np.sqrt(np.maximum(m, 2.0 ** -16)))).max(axis=2)
        out.append(np.nanmax(tile_view(e, H, W), axis=2))
    return n, out


@pytest.mark.gpu
def test_each_tile_stops_at_the_first_pass_that_meets_the_rule(rt, weekend, gpu_required):
    cam = rt.default_camera(120)
    initial, max_samples, seed, thr = 4, 256, 21, 4 * LEVEL
    acc, err, _ = rt.render_adaptive(weekend, cam, max_samples=max_samples, threshold=thr, initial_samples=initial, seed=seed)
    counts = tile_counts(acc, (0, cam.image_height))
    n, e = expected_tile_errors(rt, weekend, cam, initial, max_samples, seed)
    stop = np.full(counts.shape, n[-1])
    last_e = e[-1].copy()
    decided = np.zeros(counts.shape, bool)
    close = np.zeros(counts.shape, bool)
    for k in range(1, len(n)):
        ek = e[k - 1]
        live = ~decided
        close |= live & (np.abs(ek - thr) <= 1e-4 * thr)          # f32 kernel vs f64 here: too close to call
        now = live & (ek <= thr)
        stop[now], last_e[now] = n[k], ek[now]
        decided |= now
    ok = ~close
    assert ok.mean() > 0.95
    assert np.array_equal(counts[ok], stop[ok])
    assert len(set(counts.ravel().tolist())) >= 3                # the threshold really splits the frame
    np.testing.assert_allclose(err[ok], last_e[ok], rtol=1e-5, atol=1e-9)


@pytest.mark.gpu
def test_rgb8_output_and_stats(rt, weekend, gpu_required):
    F = rt._ffi
    cam = rt.default_camera(100)
    H, W = cam.image_height, cam.image_width
    p = F.RenderParams(seed=9, max_depth=50, row_begin=3, row_end=60, device=-1, flags=F.FLAG_COUNT_TRAVERSAL)
    ad = F.AdaptiveParams(initial_samples=8, max_samples=128, threshold=LEVEL)
    acc = np.empty((H, W, 4), np.float32)
    rgb = np.empty((H, W, 3), np.uint8)
    err = np.empty(((H + 3) // 4, (W + 7) // 8), np.float32)
    st = F.Stats()
    F.check(F.lib.b200rt_render_adaptive(weekend.device(), C.byref(cam), C.byref(p), C.byref(ad), acc.ctypes.data, rgb.ctypes.data,
                                         err.ctypes.data, C.byref(st)))
    assert np.array_equal(rgb, rt.resolve_rgb8(acc, samples=0))
    assert st.paths == int(acc[..., 3].sum()) and st.rays > st.paths and st.node_visits > 0
    assert st.kernel_ms > 0 and st.total_ms >= st.kernel_ms and st.launches >= 3
    acc2, err2, _ = rt.render_adaptive(weekend, cam, 128, LEVEL, 8, seed=9, rows=(3, 60), count_traversal=True)
    assert np.array_equal(acc2, acc) and np.array_equal(err2, err)
    # every output is optional
    F.check(F.lib.b200rt_render_adaptive(weekend.device(), C.byref(cam), C.byref(p), C.byref(ad), None, None, None, None))


def block_stats(img, ref, b=10):
    H, W = ref.shape[:2]
    d = (img - ref)[: H - H % b, : W - W % b]
    d = d.reshape(H // b, b, W // b, b, -1)
    rmse = np.sqrt((d ** 2).mean(axis=(1, 3, 4))).ravel()
    bias = d.mean(axis=(1, 3, 4)).ravel()
    return rmse, bias


# Chosen on one B200 (scripts/adaptive_probe.py, profiles/adaptive_probe.json): these settings meet every criterion below with
# a margin of 8-15 % at this seed and at two others
QUALITY_MAX, QUALITY_LEVELS, QUALITY_SEED = 1024, 1.0, 77


@pytest.mark.gpu
def test_adaptive_beats_uniform_at_equal_samples(rt, gpu_required):
    g = np.load(os.path.join(GOLDEN, "weekend_mean_300x200_4096spp.npz"))
    gamma = lambda x: np.sqrt(np.clip(x, 0.0, 1.0))
    ref = gamma(0.5 * (g["mean_a"].astype(np.float64) + g["mean_b"]))
    scene = rt.Scene.from_json(open(os.path.join(GOLDEN, "weekend_scene.json")).read(), 0x5EED)
    cam = rt.default_camera(300)
    acc, _, st = rt.render_adaptive(scene, cam, QUALITY_MAX, QUALITY_LEVELS * LEVEL, 16, seed=QUALITY_SEED)
    spp = int(np.ceil(st.paths / (cam.image_width * cam.image_height)))      # the uniform frame gets at least as many samples
    uni, _ = rt.render(scene, cam, samples=spp, seed=QUALITY_SEED)
    a = gamma(acc[..., :3].astype(np.float64) / acc[..., 3:4])
    u = gamma(uni[..., :3].astype(np.float64) / spp)
    rmse = lambda x: float(np.sqrt(np.mean((x - ref) ** 2)))
    ra, ba = block_stats(a, ref)
    ru, bu = block_stats(u, ref)
    worst = lambda r: float(np.sort(r)[-len(r) // 10:].mean())
    print(f"adaptive {st.paths / a[..., 0].size:.1f} spp vs uniform {spp}: rmse {rmse(a):.5f} / {rmse(u):.5f}, "
          f"worst decile {worst(ra):.5f} / {worst(ru):.5f}, block |bias| max {np.abs(ba).max():.5f} / {np.abs(bu).max():.5f}")
    assert rmse(a) <= rmse(u)
    assert worst(ra) < worst(ru)
    assert np.abs(ba).max() <= np.abs(bu).max() and np.sqrt(np.mean(ba ** 2)) <= np.sqrt(np.mean(bu ** 2))


@pytest.mark.gpu
def test_invalid_arguments(rt, weekend, gpu_required):
    F = rt._ffi
    cam = rt.default_camera(64)
    dev = weekend.device()

    def call(scene=dev, camera=C.byref(cam), initial=4, max_samples=16, thr=0.01, flags=0, shard=0):
        p = F.RenderParams(seed=1, max_depth=8, flags=flags, shard_count=shard, device=-1)
        ad = F.AdaptiveParams(initial_samples=initial, max_samples=max_samples, threshold=thr)
        rc = F.lib.b200rt_render_adaptive(scene, camera, C.byref(p), C.byref(ad), None, None, None, None)
        return rc, F.lib.b200rt_last_error().decode()

    assert call()[0] == F.OK
    for kw, msg in [(dict(flags=F.FLAG_ACCUMULATE), "ACCUMULATE"), (dict(shard=2), "shard_count"), (dict(initial=0), "initial_samples"),
                    (dict(max_samples=4), "max_samples"), (dict(thr=-0.1), "threshold"), (dict(thr=float("nan")), "threshold"),
                    (dict(thr=float("inf")), "threshold"), (dict(scene=None), "NULL"), (dict(camera=None), "NULL")]:
        rc, err = call(**kw)
        assert rc == F.EINVAL and msg in err, (kw, rc, err)
    ad, p = F.AdaptiveParams(4, 16, 0.01), F.RenderParams(device=-1)
    for params, adaptive in ((None, C.byref(ad)), (C.byref(p), None)):
        rc = F.lib.b200rt_render_adaptive(dev, C.byref(cam), params, adaptive, None, None, None, None)
        assert rc == F.EINVAL and "NULL" in F.lib.b200rt_last_error().decode()


@pytest.mark.gpu
def test_concurrent_adaptive_and_plain_renders(rt, weekend, gpu_required):
    cam = rt.default_camera(160)
    want_a = rt.render_adaptive(weekend, cam, 64, LEVEL, 4, seed=5)[0]
    want_p = rt.render(weekend, cam, samples=24, seed=6)[0]
    got, errors = {"a": [], "p": []}, []

    def run(kind):
        try:
            for _ in range(4):
                got[kind].append(rt.render_adaptive(weekend, cam, 64, LEVEL, 4, seed=5)[0] if kind == "a"
                                 else rt.render(weekend, cam, samples=24, seed=6)[0])
        except Exception as e:   # surfaced below
            errors.append(e)

    threads = [threading.Thread(target=run, args=(k,)) for k in ("a", "p", "a")]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    assert len(got["a"]) == 8 and all(np.array_equal(x, want_a) for x in got["a"])
    assert len(got["p"]) == 4 and all(np.array_equal(x, want_p) for x in got["p"])


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.check_call(["make", "-C", ROOT, "cli"], stdout=subprocess.DEVNULL)
    return lambda *a: subprocess.run([CLI, *a], capture_output=True, text=True, cwd=ROOT)


def test_cli_rejects_adaptive_with_gpus_or_checkpoint(cli, tmp_path):
    for extra in (["--gpus", "2"], ["--checkpoint", str(tmp_path / "c.ckpt")], [], ["--adaptive-initial", "0"]):
        args = ["render", "random", "-w", "40", "-s", "8", "-o", str(tmp_path / "x.png")] + extra
        args += ["--adaptive", "-1" if not extra else "1"]
        r = cli(*args)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr)
    assert not (tmp_path / "x.png").exists() and not (tmp_path / "c.ckpt").exists()


@pytest.mark.gpu
def test_cli_adaptive_png_equals_the_api(rt, cli, tmp_path, gpu_required):
    from PIL import Image
    png = tmp_path / "a.png"
    r = cli("-v", "render", "random", "-w", "300", "-s", "256", "--adaptive", "1", "--seed", "5", "-o", str(png))
    assert r.returncode == 0, r.stderr
    assert "spp on average" in r.stderr and "passes" in r.stderr
    acc, _, _ = rt.render_adaptive(rt.Scene.named("random", seed=5), rt.default_camera(300), 256, 1.0 / 255.0, 16, seed=5)
    assert np.array_equal(np.asarray(Image.open(png).convert("RGB")), rt.resolve_rgb8(acc, samples=0))
