"""PackRGB on the GPU: RGB24 and RGB30 packed into one GRAY32 plane in Qt's QImage layouts, checked against a numpy restatement of
the bit layout on fixture images and on noise at widths that exercise the row tails and the 16-pixel vectors, in device batches,
in fused chains that download one 4-byte plane, and from 16 host threads on one handle."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
import vapoursynth_zip_b200 as vz
from clahe_ref import clahe_plane
from helpers import assert_same_planes, noise_clip, to_node
from oracle import fixtures as fx

pytestmark = pytest.mark.gpu


def pack24(r, g, b):
    u = lambda p: p.astype(np.uint32)
    return (np.uint32(0xFF) << np.uint32(24)) | (u(r) << np.uint32(16)) | (u(g) << np.uint32(8)) | u(b)


def pack30(r, g, b):
    c = lambda p: np.minimum(p.astype(np.uint32), np.uint32(1023))
    return np.uint32(0xC0000000) | (c(r) << np.uint32(20)) | (c(g) << np.uint32(10)) | c(b)


def rgb30_clip(w, h, seed, wide=True):
    """RGB30 planes: 16-bit noise narrowed to 10 bits; with `wide`, about one sample in eight of each plane set to a value from
    1024 to 65535, which the clamp must keep inside its own field."""
    planes = [p >> 6 for p in noise_clip("RGB48", w, h, seed=seed)["planes"]]
    if wide:
        rng = np.random.default_rng(seed + 1)
        for p in planes:
            m = rng.random(p.shape) < 0.125
            p[m] = rng.integers(1024, 65536, size=int(m.sum()), dtype=np.uint64).astype(np.uint16)
        assert all(int(p.max()) > 1023 for p in planes if p.size >= 64)
    return {"format": "RGB30", "planes": planes}


def packed(frame):
    assert frame.format is vz.GRAY32 and len(frame.planes) == 1
    return np.ascontiguousarray(frame.planes[0])


@pytest.mark.parametrize("geo", ["full", "odd", "tiny"])
def test_rgb24_fixtures(geo):
    src = fx.make_clip("RGB24", geo)
    r, g, b = src["planes"]
    got = packed(to_node(src).vszip.PackRGB().get_frame(0))
    assert_same_planes([got], [pack24(r, g, b)], f"RGB24 {geo}")
    # on a little-endian host the words are the bytes B, G, R, 255: what QImage::Format_RGB32 reads
    want = np.stack([b, g, r, np.full_like(r, 255)], axis=-1)
    assert np.array_equal(got.view(np.uint8).reshape(want.shape), want)


@pytest.mark.parametrize("w", [1, 15, 16, 17, 33, 1919])
@pytest.mark.parametrize("fmt", ["RGB24", "RGB30"])
def test_noise_widths(fmt, w):
    h = 37
    src = noise_clip("RGB24", w, h, seed=w) if fmt == "RGB24" else rgb30_clip(w, h, seed=w)
    got = packed(to_node(src).vszip.PackRGB().get_frame(0))
    want = (pack24 if fmt == "RGB24" else pack30)(*src["planes"])
    assert_same_planes([got], [want], f"{fmt} noise {w}x{h}")


def test_rgb30_clamp_and_top_bits():
    """Every field at its largest and over it, each plane alone, in the vector part and in the tail of a row."""
    w, h = 20, 4
    vals = np.array([0, 1, 1023, 1024, 0x3FF | 0x400, 0xFFFF], np.uint16)
    planes = [np.zeros((h, w), np.uint16) for _ in range(3)]
    for c in range(3):
        planes[c][c, :len(vals)] = vals
        planes[c][c, 16:16 + 4] = vals[2:]
    got = packed(to_node({"format": "RGB30", "planes": planes}).vszip.PackRGB().get_frame(0))
    assert_same_planes([got], [pack30(*planes)], "RGB30 edge values")
    assert int(got[0, 3]) == 0xC0000000 | 1023 << 20 and int(got[1, 5]) == 0xC0000000 | 1023 << 10 and int(got[2, 19]) == 0xC00003FF
    assert (got >> np.uint32(30) == 3).all()


def test_props():
    src = noise_clip("RGB24", 64, 36, seed=1)
    node = vz.core.clip_from_frames("RGB24", [src["planes"]], props={"_ColorRange": 0, "_Matrix": 0, "x": 3})
    assert node.vszip.PackRGB().get_frame(0).props == {"_ColorRange": 0, "_Matrix": 0, "x": 3}


def test_rgb24_device_batch_sub_range():
    w, h, n = 1920, 1080, 12
    a, d = vz.DeviceClip("RGB24", w, h, n), vz.DeviceClip("GRAY32", w, h, n)
    a.fill_noise(seed=9)
    d.fill_noise(seed=10)  # frames outside the range must keep these
    outside = {i: d.download(i)[0] for i in (2, 10)}
    f = vz.PackRGBFilter(a.info())
    f.run_device(a, d, first=3, count=7)
    vz.core.sync()
    for i in range(3, 10):
        assert_same_planes(d.download(i), [pack24(*a.download(i))], f"1080p RGB24 frame {i}")
    for i, p in outside.items():
        assert_same_planes(d.download(i), [p], f"frame {i} outside the range")
    with pytest.raises(vz.Error, match="^PackRGB: device clip does not match the format the filter was created for$"):
        f.run_device(a, a)
    wrong = vz.DeviceClip("GRAY16", w, h, n)
    with pytest.raises(vz.Error, match="^PackRGB: device clip does not match the format the filter was created for$"):
        f.run_device(a, wrong)


def test_4k_rgb30_device_batch():
    w, h, n = 3840, 2160, 3
    a, d = vz.DeviceClip("RGB30", w, h, n), vz.DeviceClip("GRAY32", w, h, n)
    for i in range(n):
        a.upload(i, rgb30_clip(w, h, seed=70 + i)["planes"])
    vz.PackRGBFilter(a.info()).run_device(a, d)
    vz.core.sync()
    for i in range(n):
        assert_same_planes(d.download(i), [pack30(*a.download(i))], f"4K RGB30 frame {i}")


def _fused_and_plain(src, build):
    vz.core.fuse_chains = True
    try:
        node = build(to_node(src))
        before = vz.core.transfer_bytes()
        fused = node.get_frame(0)
        after = vz.core.transfer_bytes()
        assert getattr(node, "_chain", None) is not None, "the chain was not fused"
    finally:
        vz.core.fuse_chains = False
    try:
        plain = build(to_node(src)).get_frame(0)
    finally:
        vz.core.fuse_chains = True
    assert_same_planes(fused.planes, plain.planes, "fused vs unfused")
    assert fused.format is plain.format and fused.props == plain.props, (fused.props, plain.props)
    return fused, (after[0] - before[0], after[1] - before[1])


def test_gray8_boxblur_clahe_colormap_packrgb_chain():
    cv2 = pytest.importorskip("cv2")
    src = fx.make_clip("GRAY8", "odd")
    y = src["planes"][0]
    fused, moved = _fused_and_plain(src, lambda c: c.vszip.BoxBlur(hradius=2, vradius=2).vszip.CLAHE(limit=3).vszip.ColorMap(2)
                                    .vszip.PackRGB())
    assert moved == (y.size, 4 * y.size)
    rgb = cv2.applyColorMap(clahe_plane(oracle.boxblur_plane(y, 2, 1, 2, 1), 8, 3, (3, 3)), 2)[..., ::-1]
    assert_same_planes([packed(fused)], [pack24(rgb[..., 0], rgb[..., 1], rgb[..., 2])], "BoxBlur -> CLAHE -> ColorMap -> PackRGB")


def test_rgb30_limiter_packrgb_chain():
    w, h = 642, 361
    src = rgb30_clip(w, h, seed=21)
    lo, hi = [64, 100, 0], [940, 1023, 600]
    fused, moved = _fused_and_plain(src, lambda c: c.vszip.Limiter(min=lo, max=hi).vszip.PackRGB())
    assert moved == (6 * w * h, 4 * w * h)
    want = pack30(*[np.clip(p, a, b) for p, a, b in zip(src["planes"], lo, hi)])
    assert_same_planes([packed(fused)], [want], "RGB30 Limiter -> PackRGB")


def test_one_handle_many_threads():
    frames = 24
    clips = [rgb30_clip(322, 182, seed=900 + i) for i in range(frames)]
    want = [pack30(*c["planes"]) for c in clips]
    node = vz.core.clip_from_frames("RGB30", [c["planes"] for c in clips]).vszip.PackRGB()
    order = [(i * 7) % frames for i in range(frames * 3)]
    with ThreadPoolExecutor(16) as ex:
        results = list(ex.map(lambda n: (n, node.get_frame(n)), order))
    for n, fr in results:
        assert_same_planes([packed(fr)], [want[n]], f"PackRGB frame {n}")
