"""The feature-guided à-trous denoiser (b200rt_render_denoised, b200rt_denoise, rt.render_denoised, rt.denoise, ray-cli --denoise).

Deterministic checks first: the noisy buffer is a plain render bit for bit, the features are the first hits of the render's own
primary rays (rebuilt here from the RNG, camera and closest-hit hooks), the denoised frame is the filter applied to two plain
half renders, and the filter matches a float64 restatement of csrc/denoise_plan.hpp.  The quality checks run at a fixed seed."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
CLI = os.path.join(ROOT, "ray-cli")
B3 = {-2: 1 / 16, -1: 1 / 4, 0: 3 / 8, 1: 1 / 4, 2: 1 / 16}
G3 = {-1: 0.25, 0: 0.5, 1: 0.25}
EPS_A, SIGMA_L, EPS_L, SIGMA_N, SIGMA_Z, SIGMA_A = 1e-3, 4.0, 1e-10, 128.0, 0.05, 0.1


def lum(y):
    return 0.2126 * y[..., 0] + 0.7152 * y[..., 1] + 0.0722 * y[..., 2]


def filter_f64(A, B, feat, iterations):
    """csrc/denoise_plan.hpp in float64."""
    A, B, feat = A.astype(np.float64), B.astype(np.float64), feat.astype(np.float64)
    H, W = A.shape[:2]
    N, Z, alb = feat[0, ..., :3], feat[0, ..., 3], np.maximum(feat[1, ..., :3], EPS_A)
    na, nb = A[..., 3], B[..., 3]
    n = na + nb
    x = (A[..., :3] + B[..., :3]) / n[..., None] / alb
    la, lb = lum(A[..., :3] / na[..., None] / alb), lum(B[..., :3] / nb[..., None] / alb)
    v = (la - lb) ** 2 * na * nb / n ** 2
    miss = Z == 0
    ys, xs = np.arange(H), np.arange(W)
    for i in range(iterations):
        s = 2 ** i
        vp = np.pad(v, 1, mode="edge")
        vbar = sum(G3[dy] * G3[dx] * vp[1 + dy:1 + dy + H, 1 + dx:1 + dx + W] for dy in (-1, 0, 1) for dx in (-1, 0, 1))
        lp, lscale = lum(x), SIGMA_L * np.sqrt(vbar) + EPS_L
        sw, sx, sv = np.zeros((H, W)), np.zeros((H, W, 3)), np.zeros((H, W))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                qy, qx = ys + dy * s, xs + dx * s
                ok = ((qy >= 0) & (qy < H))[:, None] & ((qx >= 0) & (qx < W))[None, :]
                Y, X = np.clip(qy, 0, H - 1)[:, None], np.clip(qx, 0, W - 1)[None, :]
                xq, vq, Nq, Zq, aq = x[Y, X], v[Y, X], N[Y, X], Z[Y, X], alb[Y, X]
                w = np.full((H, W), B3[dx] * B3[dy])
                if dx or dy:
                    nn = np.sqrt((N ** 2).sum(-1) * (Nq ** 2).sum(-1))
                    c = np.where(nn > 0, np.minimum((N * Nq).sum(-1) / np.where(nn > 0, nn, 1), 1.0), 0.0)
                    zm = np.maximum(Z, Zq)
                    e = (np.exp(-np.abs(lp - lum(xq)) / lscale) * np.where(c > 0, np.maximum(c, 0) ** SIGMA_N, 0.0)
                         * np.where(zm > 0, np.exp(-np.abs(Z - Zq) / (SIGMA_Z * np.where(zm > 0, zm, 1) * s * max(abs(dx), abs(dy)))), 1.0)
                         * np.exp(-np.abs(feat[1, ..., :3] - feat[1][Y, X, :3]).sum(-1) / SIGMA_A))
                    w = w * np.where(miss != (Zq == 0), 0.0, e)
                w = np.where(ok, w, 0.0)
                sw += w; sx += w[..., None] * xq; sv += w * w * vq
        x = np.where(miss[..., None], x, sx / sw[..., None])
        v = np.where(miss, v, sv / sw ** 2)
    out = np.concatenate([x * alb * n[..., None], n[..., None]], axis=-1)
    out[miss] = (A + B)[miss]
    return out


def synthetic(H=24, W=37, seed=0):
    """Two noisy halves of a scene of three planes, a sphere-like bump, a sky region and a textured albedo."""
    rng = np.random.default_rng(seed)
    feat = np.zeros((2, H, W, 4), np.float32)
    yy, xx = np.mgrid[0:H, 0:W]
    nrm = np.zeros((H, W, 3))
    nrm[..., 1] = 1.0
    nrm[:, W // 2:] = (0.0, 0.0, -1.0)
    bump = (yy - H / 2) ** 2 + (xx - W / 3) ** 2 < 20
    nrm[bump] = np.stack([(xx - W / 3)[bump], np.full(bump.sum(), 3.0), (yy - H / 2)[bump]], 1)
    nrm /= np.linalg.norm(nrm, axis=-1, keepdims=True)
    feat[0, ..., :3] = nrm
    feat[0, ..., 3] = np.where(xx < W // 2, 5.0 + 0.05 * yy, 9.0)
    feat[0, bump, 3] = 4.0
    sky = yy >= H - 4
    feat[0, sky] = 0.0
    feat[1, ..., :3] = np.stack([0.2 + 0.6 * ((xx // 4 + yy // 4) % 2), 0.3 + 0.02 * xx, np.full((H, W), 0.5)], -1)
    feat[1, sky, :3] = (0.6, 0.7, 1.0)
    feat[1, 0, :3] = 0.0                                   # a black row: the albedo floor
    E = 0.5 + 0.3 * (xx < W // 2)
    A = np.zeros((H, W, 4), np.float32)
    B = np.zeros((H, W, 4), np.float32)
    for buf, k in ((A, 8), (B, 9)):
        buf[..., :3] = feat[1, ..., :3] * (E * rng.gamma(4.0, 0.25, (k, H, W)).sum(0))[..., None]
        buf[..., 3] = k
    return A, B, feat


@pytest.fixture(scope="module")
def lensless(rt):
    return lambda width: rt.camera((13.0, 2.0, 3.0), (0.0, 0.0, 0.0), vfov=20.0, aperture=None, width=width)


# ---- the filter alone ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("iterations", [1, 3, 5])
def test_filter_matches_float64_restatement(rt, gpu_required, iterations):
    A, B, feat = synthetic(seed=iterations)
    got = rt.denoise(A, B, feat, iterations=iterations)
    want = filter_f64(A, B, feat, iterations)
    assert np.array_equal(got[..., 3], want[..., 3])
    np.testing.assert_allclose(got[..., :3], want[..., :3], rtol=1e-4, atol=1e-6)
    sky = feat[0, ..., 3] == 0
    assert np.array_equal(got[sky], (A + B)[sky])          # miss pixels are untouched
    assert not np.allclose(got[~sky, :3], (A + B)[~sky, :3], rtol=1e-3)   # and the others are filtered


@pytest.mark.gpu
def test_constant_image_is_returned_unchanged(rt, gpu_required):
    H, W = 20, 30
    A = np.zeros((H, W, 4), np.float32)
    A[...] = (0.7 * 6, 0.25 * 6, 1.3 * 6, 6)
    _, _, feat = synthetic(H, W, seed=4)
    feat[0, ..., 3] = np.maximum(feat[0, ..., 3], 1.0)      # no sky
    out = rt.denoise(A, A, feat, iterations=5)
    np.testing.assert_allclose(out, A + A, rtol=1e-6)


@pytest.mark.gpu
def test_no_leakage_across_an_albedo_step(rt, gpu_required):
    H, W, k = 64, 64, 8
    rng = np.random.default_rng(12)
    feat = np.zeros((2, H, W, 4), np.float32)
    feat[0, ..., 2], feat[0, ..., 3] = -1.0, 5.0
    red, blue = np.array([0.8, 0.1, 0.1]), np.array([0.1, 0.1, 0.8])
    feat[1, :, : W // 2, :3], feat[1, :, W // 2:, :3] = red, blue
    halves = []
    for _ in range(2):
        a = np.zeros((H, W, 4), np.float32)
        a[..., :3] = feat[1, ..., :3] * rng.gamma(2.0, 0.5, (k, H, W)).sum(0)[..., None]
        a[..., 3] = k
        halves.append(a)
    out = rt.denoise(*halves, feat, iterations=5)
    noisy = (halves[0][..., :3] + halves[1][..., :3]) / (2 * k)
    den = out[..., :3] / out[..., 3:]
    for col, side in ((W // 2 - 1, slice(0, W // 2)), (W // 2, slice(W // 2, W))):
        mean = noisy[:, side].reshape(-1, 3).mean(0)
        se = noisy[:, side].reshape(-1, 3).std(0) / np.sqrt(H)
        assert np.all(np.abs(den[:, col].mean(0) - mean) <= 3 * se), (col, den[:, col].mean(0), mean, se)


# ---- the renderer -----------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 17, 64])
def test_accum_is_the_plain_render(rt, weekend, gpu_required, n):
    cam = rt.default_camera(150)                              # 150 x 100: a ragged last tile column
    den, acc, feat, st = rt.render_denoised(weekend, cam, n, feature_samples=min(4, n), seed=3, sample_offset=5)
    plain, pst = rt.render(weekend, cam, samples=n, seed=3, sample_offset=5)
    assert np.array_equal(acc, plain)
    assert st.paths == pst.paths == n * 150 * 100 and st.rays == pst.rays
    assert st.kernel_ms > 0 and st.total_ms >= st.kernel_ms and st.launches >= 10
    assert np.array_equal(den[..., 3], plain[..., 3]) and np.all(np.isfinite(den))


def expected_features(rt, scene, cam, seed, k, sample_offset=0):
    """Each field of the features summed over the k primary rays in sample order in f32 and divided by k, from the hooks."""
    H, W = cam.image_height, cam.image_width
    desc = scene.desc.contents
    nz = np.zeros((H * W, 4), np.float32)
    al = np.zeros((H * W, 3), np.float32)
    kinds = np.array([desc.materials[i].kind for i in range(desc.n_prims)])
    texs = np.array([desc.materials[i].texture for i in range(desc.n_prims)])
    pix = np.arange(H * W)
    px, py = (pix % W).astype(np.float32), (pix // W).astype(np.float32)
    for s in range(k):
        u = np.array([rt.rng_uniforms(seed, int(p), sample_offset + s, 2) for p in pix], np.float32)
        xy = np.stack([px + u[:, 0], py + u[:, 1]], 1)
        rays = rt.camera_rays(cam, xy)
        ids, hits, _ = rt.closest_hit(scene, rays, 0.001, float("inf"))
        hit = ids >= 0
        d = rays[:, 3:6]
        depth = hits["t"] * np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
        f = np.zeros((H * W, 4), np.float32)
        f[hit, :3], f[hit, 3] = hits["n"][hit], depth[hit]
        a = np.zeros((H * W, 3), np.float32)
        kind = np.where(hit, kinds[np.maximum(ids, 0)], -1)
        for i in np.nonzero(kind == rt._ffi.MAT_METAL)[0]:
            a[i] = tuple(desc.materials[ids[i]].albedo)
        a[kind == rt._ffi.MAT_DIELECTRIC] = 1.0
        texd = np.isin(kind, [rt._ffi.MAT_LAMBERTIAN, rt._ffi.MAT_DIFFUSE_LIGHT, rt._ffi.MAT_FAIRY_LIGHT])
        tex = texs[np.maximum(ids, 0)]
        for t in sorted(set(tex[texd].tolist())):
            sel = texd & (tex == t)
            h = hits[sel]
            a[sel] = rt.texture_value(scene, t, np.column_stack([h["u"], h["v"], h["p"]]))
        if (~hit).any():                                       # a miss record returns the device's background(d)
            sky = np.zeros((~hit).sum(), rt.HIT_DTYPE)
            sky["id"] = -1
            a[~hit] = rt.scatter(scene, rays[~hit], sky)["emitted"]
        nz, al = nz + f, al + a
    kf = np.float32(k)
    return (nz / kf).reshape(H, W, 4), (al / kf).reshape(H, W, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 4])
def test_features_are_the_first_hits_of_the_primary_rays(rt, weekend, lensless, gpu_required, k):
    cam = lensless(48)
    seed = 8
    _, _, feat, _ = rt.render_denoised(weekend, cam, 8, feature_samples=k, seed=seed)
    nz, al = expected_features(rt, weekend, cam, seed, k)
    assert np.array_equal(feat[0], nz)
    assert np.array_equal(feat[1][..., :3], al) and np.all(feat[1][..., 3] == 0)
    # pixels with feature rays on geometry and pixels whose feature rays all met the sky are both there
    sky = feat[0, ..., 3] == 0
    assert (~sky).mean() > 0.5 and sky.any() and np.all((feat[1][sky][:, :3] > 0.4) & (feat[1][sky][:, :3] <= 1.0))


@pytest.mark.gpu
def test_denoised_is_the_filter_of_two_plain_halves(rt, weekend, gpu_required):
    cam = rt.default_camera(120)
    n, seed, off = 33, 4, 3
    den, acc, feat, _ = rt.render_denoised(weekend, cam, n, feature_samples=3, iterations=4, seed=seed, sample_offset=off)
    a, _ = rt.render(weekend, cam, samples=n // 2, seed=seed, sample_offset=off)
    b, _ = rt.render(weekend, cam, samples=n - n // 2, seed=seed, sample_offset=off + n // 2)
    assert np.array_equal(den, rt.denoise(a, b, feat, iterations=4))
    rgb = np.empty(acc.shape[:2] + (3,), np.uint8)
    F = rt._ffi
    p = F.RenderParams(samples=n, sample_offset=off, max_depth=50, seed=seed, device=-1)
    dn = F.DenoiseParams(feature_samples=3, iterations=4)
    F.check(F.lib.b200rt_render_denoised(weekend.device(), C.byref(cam), C.byref(p), C.byref(dn), None, None, None, rgb.ctypes.data, None))
    assert np.array_equal(rgb, rt.resolve_rgb8(den, samples=0))


@pytest.mark.gpu
def test_invalid_arguments(rt, weekend, gpu_required):
    F = rt._ffi
    cam = rt.default_camera(64)
    dev = weekend.device()

    def call(scene=dev, camera=C.byref(cam), samples=8, k=4, it=5, flags=0, shard=0, rows=(0, 0), params=True, dn=True):
        p = F.RenderParams(samples=samples, seed=1, max_depth=8, flags=flags, shard_count=shard, row_begin=rows[0], row_end=rows[1], device=-1)
        d = F.DenoiseParams(feature_samples=k, iterations=it)
        rc = F.lib.b200rt_render_denoised(scene, camera, C.byref(p) if params else None, C.byref(d) if dn else None,
                                          None, None, None, None, None)
        return rc, F.lib.b200rt_last_error().decode()

    assert call()[0] == F.OK and call(rows=(0, cam.image_height))[0] == F.OK
    for kw, msg in [(dict(samples=1, k=1), "samples"), (dict(k=0), "feature_samples"), (dict(k=9), "feature_samples"),
                    (dict(it=0), "iterations"), (dict(it=6), "iterations"), (dict(flags=F.FLAG_ACCUMULATE), "ACCUMULATE"),
                    (dict(shard=2), "shard_count"), (dict(rows=(0, 10)), "row range"), (dict(rows=(4, 0)), "row range"),
                    (dict(scene=None), "NULL"), (dict(camera=None), "NULL"), (dict(params=False), "NULL"), (dict(dn=False), "NULL")]:
        rc, err = call(**kw)
        assert rc == F.EINVAL and msg in err, (kw, rc, err)
    A, B, feat = synthetic()
    for it in (0, 6):
        with pytest.raises(rt.B200rtError) as e:
            rt.denoise(A, B, feat, iterations=it)
        assert e.value.code == F.EINVAL


@pytest.mark.gpu
def test_deterministic_and_thread_safe(rt, weekend, gpu_required):
    cam = rt.default_camera(96)
    want = rt.render_denoised(weekend, cam, 12, seed=6)
    again = rt.render_denoised(weekend, cam, 12, seed=6)
    for x, y in zip(want[:3], again[:3]):
        assert x.tobytes() == y.tobytes()
    got, errors = [], []

    def run():
        try:
            for _ in range(3):
                got.append(rt.render_denoised(weekend, cam, 12, seed=6)[:3])
        except Exception as e:   # surfaced below
            errors.append(e)

    threads = [threading.Thread(target=run) for _ in range(2)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not errors, errors
    assert len(got) == 6 and all(all(x.tobytes() == y.tobytes() for x, y in zip(g, want[:3])) for g in got)


# ---- quality ------------------------------------------------------------------------------------------------------------
def gamma(x):
    return np.sqrt(np.clip(x, 0.0, 1.0))


def rmse(x, ref):
    return float(np.sqrt(np.mean((x - ref) ** 2)))


QUALITY_SEED = 101


# Measured on one NVIDIA B200 (scripts/denoise_probe.py, profiles/denoise_probe.json): denoised / noisy RMSE is 0.73-0.75 at
# 16 spp and 1.55-1.57 at 1024 spp on this frame at seeds 101, 202 and 303.  The albedo of the remodulation is the mean of
# only the feature rays, and its sampling noise enters the output directly where the ground's texture varies within a pixel.
@pytest.mark.xfail(strict=True, reason="targets 0.6x at 16 spp and 1.05x at 1024 spp not met on the Weekend frame (DESIGN.md)")
@pytest.mark.gpu
def test_quality_weekend(rt, gpu_required):
    g = np.load(os.path.join(GOLDEN, "weekend_mean_300x200_4096spp.npz"))
    ref = gamma(0.5 * (g["mean_a"].astype(np.float64) + g["mean_b"]))
    scene = rt.Scene.from_json(open(os.path.join(GOLDEN, "weekend_scene.json")).read(), 0x5EED)
    cam = rt.default_camera(300)
    for n, bound in ((16, 0.6), (1024, 1.05)):
        den, acc, _, _ = rt.render_denoised(scene, cam, n, seed=QUALITY_SEED)
        rd, rn = rmse(gamma(den[..., :3] / den[..., 3:]), ref), rmse(gamma(acc[..., :3] / n), ref)
        print(f"weekend {n} spp: denoised rmse {rd:.5f}, noisy {rn:.5f}, ratio {rd / rn:.3f}")
        assert rd <= bound * rn, (n, rd, rn)


def cornell_camera(rt, width):
    return rt.camera((278.0, 278.0, -800.0), (278.0, 278.0, 0.0), vfov=40.0, focal_length=1.0, aperture=0.00001, width=width,
                     aspect_ratio=(1, 1), focus_length=10.0)


@pytest.mark.gpu
def test_quality_cornell(rt, gpu_required):
    scene = rt.Scene.named("cornell")
    cam = cornell_camera(rt, 150)
    ref_acc, _ = rt.render(scene, cam, samples=4096, seed=QUALITY_SEED + 1)
    ref = gamma(ref_acc[..., :3].astype(np.float64) / 4096)
    for n, bound in ((16, 0.6), (1024, 1.05)):
        den, acc, _, _ = rt.render_denoised(scene, cam, n, seed=QUALITY_SEED)
        rd, rn = rmse(gamma(den[..., :3] / den[..., 3:]), ref), rmse(gamma(acc[..., :3] / n), ref)
        print(f"cornell {n} spp: denoised rmse {rd:.5f}, noisy {rn:.5f}, ratio {rd / rn:.3f}")
        assert rd <= bound * rn, (n, rd, rn)


# ---- CLI ---------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.check_call(["make", "-C", ROOT, "cli"], stdout=subprocess.DEVNULL)
    return lambda *a: subprocess.run([CLI, *a], capture_output=True, text=True, cwd=ROOT)


def test_cli_rejects_denoise_combinations(cli, tmp_path):
    for extra in (["--adaptive", "1"], ["--gpus", "2"], ["--checkpoint", str(tmp_path / "c.ckpt")], ["-s", "1"],
                  ["--denoise-features", "9"], ["--denoise-features", "0"]):
        r = cli("render", "random", "-w", "40", "-s", "8", "-o", str(tmp_path / "x.png"), "--denoise", *extra)
        assert r.returncode == 2 and "error:" in r.stderr, (extra, r.stderr)
    assert not (tmp_path / "x.png").exists() and not (tmp_path / "c.ckpt").exists()


@pytest.mark.gpu
def test_cli_denoised_png_equals_the_api(rt, cli, tmp_path, gpu_required):
    from PIL import Image
    png = tmp_path / "d.png"
    r = cli("render", "random", "-w", "200", "-s", "16", "--denoise", "--seed", "5", "-o", str(png))
    assert r.returncode == 0, r.stderr
    den, _, _, _ = rt.render_denoised(rt.Scene.named("random", seed=5), rt.default_camera(200), 16, feature_samples=4, seed=5)
    assert np.array_equal(np.asarray(Image.open(png).convert("RGB")), rt.resolve_rgb8(den, samples=0))
