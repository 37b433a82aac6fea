"""Host-side JPEG decoder (baseline and progressive) (shirley_raytracing_rs_b200/host/jpeg_decoder.cpp) — what
`image::open` / `image::load_from_memory` do for the reference's image textures
(material/texture/image_texture.rs:18-31).  Checked against PIL (libjpeg): identical bytes."""
import hashlib
import io
import os

import numpy as np
import pytest

PIL = pytest.importorskip("PIL.Image")


def _picture(w, h, seed):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    img = np.stack([127 + 120 * np.sin(x / 7.0 + seed), 127 + 120 * np.cos(y / 5.0), (x * 3 + y * 5) % 256], axis=-1)
    img += rng.normal(0, 12, size=img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


def _encode(arr, **kw):
    buf = io.BytesIO()
    PIL.fromarray(arr).save(buf, format="JPEG", **kw)
    return buf.getvalue()


def _pil_decode(data):
    return np.asarray(PIL.open(io.BytesIO(data)).convert("RGB"))


@pytest.mark.parametrize("size", [(64, 48), (1, 1), (17, 9), (33, 70), (8, 8)])
@pytest.mark.parametrize("subsampling", [0, 1, 2])      # 4:4:4 (the earth map's layout), 4:2:2, 4:2:0
@pytest.mark.parametrize("quality", [35, 90])
def test_matches_libjpeg(rt, size, subsampling, quality):
    data = _encode(_picture(*size, seed=quality + subsampling), quality=quality, subsampling=subsampling)
    got = rt.decode_jpeg(data)
    want = _pil_decode(data)
    assert got.shape == want.shape
    assert np.array_equal(got, want), np.abs(got.astype(int) - want.astype(int)).max()


@pytest.mark.parametrize("size", [(64, 48), (1, 1), (17, 9), (33, 70), (200, 120)])
@pytest.mark.parametrize("subsampling", [0, 1, 2])
@pytest.mark.parametrize("quality", [30, 92])
def test_progressive_matches_libjpeg(rt, size, subsampling, quality):
    """SOF2: spectral selection + successive approximation (DC/AC first and refinement scans, EOB runs)."""
    data = _encode(_picture(*size, seed=quality + subsampling), quality=quality, subsampling=subsampling, progressive=True)
    assert b"\xff\xc2" in data
    got = rt.decode_jpeg(data)
    want = _pil_decode(data)
    assert got.shape == want.shape
    assert np.array_equal(got, want), np.abs(got.astype(int) - want.astype(int)).max()


def test_progressive_grayscale_and_restarts(rt):
    g = _picture(90, 61, 5)[..., 0]
    data = _encode(g, quality=70, progressive=True)
    assert np.array_equal(rt.decode_jpeg(data), _pil_decode(data))
    rgb = _picture(130, 77, 6)
    for kw in ({"restart_marker_blocks": 2}, {"restart_marker_rows": 1}, {"optimize": True}):
        try:
            data = _encode(rgb, quality=60, progressive=True, **kw)
        except TypeError:
            continue
        assert np.array_equal(rt.decode_jpeg(data), _pil_decode(data)), kw


def test_grayscale_restart_and_optimized_tables(rt):
    g = _picture(50, 37, 3)[..., 0]
    data = _encode(g, quality=80)
    assert np.array_equal(rt.decode_jpeg(data), _pil_decode(data))
    rgb = _picture(120, 70, 4)
    for kw in ({"optimize": True}, {"restart_marker_blocks": 3}, {"restart_marker_rows": 1}):
        try:
            data = _encode(rgb, quality=75, **kw)
        except TypeError:
            continue
        assert np.array_equal(rt.decode_jpeg(data), _pil_decode(data)), kw


def test_rejects_bad_input(rt):
    with pytest.raises(rt.B200rtError):
        rt.decode_jpeg(b"not a jpeg at all")
    good = _encode(_picture(32, 32, 1), quality=80)
    with pytest.raises(rt.B200rtError):
        rt.decode_jpeg(good[: len(good) // 3])          # truncated before the scan


def _with_dht(bits, vals=b""):
    """A minimal stream: SOI, one DHT segment with the given 16 code-length counts, EOI."""
    seg = bytes([0x00]) + bytes(bits) + bytes(vals)
    return b"\xff\xd8" + b"\xff\xc4" + (len(seg) + 2).to_bytes(2, "big") + seg + b"\xff\xd9"


def test_rejects_oversubscribed_huffman_table(rt):
    """A DHT whose code lengths are not a prefix code (255 codes of length 1) used to index the canonical-code
    look-up table out of bounds; libjpeg calls this a bogus Huffman table."""
    bits = [255] + [0] * 15
    with pytest.raises(rt.B200rtError, match="over-subscribed"):
        rt.decode_jpeg(_with_dht(bits, bytes(255)))
    bits = [0, 0, 0, 0, 0, 0, 0, 0, 200] + [0] * 7     # 200 nine-bit codes do fit (<= 512), 3 one-bit codes never do
    with pytest.raises(rt.B200rtError):
        rt.decode_jpeg(_with_dht(bits, bytes(200)))    # valid table, but no frame: still an error, not a crash
    with pytest.raises(rt.B200rtError, match="over-subscribed"):
        rt.decode_jpeg(_with_dht([3] + [0] * 15, bytes(3)))
    with pytest.raises(rt.B200rtError):
        rt.decode_jpeg(b"\xff\xd8\xff\xda\x00\x02\xff\xd9")   # SOS with an empty body


def test_mutated_streams_never_crash(rt):
    """Byte-flip fuzzing of valid baseline and progressive streams: every outcome is an image or an error."""
    rng = np.random.default_rng(7)
    for kw in ({"quality": 80}, {"quality": 60, "progressive": True}, {"quality": 70, "optimize": True}):
        good = bytearray(_encode(_picture(40, 24, 3), **kw))
        for _ in range(150):
            bad = bytearray(good)
            for _ in range(int(rng.integers(1, 4))):
                bad[int(rng.integers(2, len(bad)))] = int(rng.integers(0, 256))
            try:
                out = rt.decode_jpeg(bytes(bad))
                assert out.ndim == 3 and out.shape[2] == 3
            except rt.B200rtError:
                pass


def test_image_path_texture_is_decoded_at_finalize(rt, tmp_path):
    """TextureLoader::ImagePath(path) -> image::open(path) at SceneBuilder::finalize (loader.rs:47-60)."""
    arr = _picture(40, 20, 9)
    path = tmp_path / "tex.jpg"
    path.write_bytes(_encode(arr, quality=95, subsampling=0))
    b = rt.SceneBuilder()
    b.add(rt.Sphere((0, 0, 0), 1.0), rt.Lambertian(rt.TextureLoader.ImagePath(str(path))))
    scene = b.finalize()
    d = scene.desc.contents
    assert d.n_images == 1 and d.images[0].width == 40 and d.images[0].height == 20
    texels = np.ctypeslib.as_array(d.images[0].rgb8, shape=(20, 40, 3))
    assert np.array_equal(texels, _pil_decode(path.read_bytes()))
    with pytest.raises(rt.B200rtError):
        b2 = rt.SceneBuilder()
        b2.add(rt.Sphere((0, 0, 0), 1.0), rt.Lambertian(rt.TextureLoader.ImagePath(str(tmp_path / "missing.jpg"))))
        b2.finalize()


def test_reference_earthmap(rt):
    """The asset the reference embeds (image_texture.rs:11): 1024x512, baseline, 4:4:4.  The package ships the same
    file (assets/README.md); the hashes pin it and its decoded texels to the reference's copy."""
    data = open(os.path.join(os.path.dirname(rt.__file__), "assets", "earthmap.jpg"), "rb").read()
    assert hashlib.sha256(data).hexdigest() == "e7c5a0062719708d0943dcc13bb48af677c46de8686e3940062f6a70285695d4"
    got = rt.decode_jpeg(data)
    assert got.shape == (512, 1024, 3)
    assert hashlib.sha256(got.tobytes()).hexdigest() == "a8cdc92a168d554ddc693785d31f5e251063724f44099571d7fbce3b43d44c45"
    assert np.array_equal(got, _pil_decode(data))
