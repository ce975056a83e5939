"""ColorMap on the GPU: bit-exact with OpenCV's applyColorMap on 8-bit luma, with the table lookup of min(x >> (bits - 8), 255) on
deeper clips, in device batches, in fused chains that upload gray and download RGB, and from 16 host threads on one handle."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
import vapoursynth_zip_b200 as vz
from clahe_ref import clahe_plane
from helpers import assert_same_planes, noise_clip, to_node
from oracle import fixtures as fx

pytestmark = pytest.mark.gpu


def table(color):
    """(256, 3) R, G, B straight from OpenCV."""
    cv2 = pytest.importorskip("cv2")
    return cv2.applyColorMap(np.arange(256, dtype=np.uint8)[:, None], color)[:, 0, ::-1]


def colormap(y, bits, color=20):
    rgb = table(color)[np.minimum(y.astype(np.uint32) >> (bits - 8), 255)]
    return [np.ascontiguousarray(rgb[..., c]) for c in range(3)]


def rgb_planes(frame):
    assert frame.format is vz.RGB24
    return [np.ascontiguousarray(p) for p in frame.planes]


@pytest.mark.parametrize("geo", ["full", "odd", "tiny"])
def test_every_map_equals_opencv_on_gray8(geo):
    cv2 = pytest.importorskip("cv2")
    src = fx.make_clip("GRAY8", geo)
    y = src["planes"][0]
    node = to_node(src)
    for k in range(22):
        want = cv2.applyColorMap(y, k)[..., ::-1]
        got = rgb_planes(node.vszip.ColorMap(k).get_frame(0))
        assert_same_planes(got, [want[..., c] for c in range(3)], f"{geo} color={k}")


@pytest.mark.parametrize(("fmt", "w", "h"), [("GRAY10", 517, 243), ("GRAY16", 517, 243), ("YUV420P10", 322, 182), ("GRAY12", 33, 7)])
def test_deep_noise_equals_the_lookup(fmt, w, h):
    bits = vz.FORMATS[fmt].bits_per_sample
    if fmt == "GRAY12":  # not an oracle fixture format: 16-bit noise narrowed to 12 bits
        src = {"format": fmt, "planes": [noise_clip("GRAY16", w, h, seed=5)["planes"][0] >> 4]}
    else:
        src = noise_clip(fmt, w, h, seed=5)
    if bits == 10:  # samples above 1023 still index the table: min(x >> 2, 255)
        wide = noise_clip("GRAY16", w, h, seed=6)["planes"][0] >> 5
        src["planes"][0] = np.where(wide >= 1024, wide, src["planes"][0]).astype(np.uint16)
        assert int(src["planes"][0].max()) > 1023
    node = to_node(src)
    for k in (0, 9, 20, 21):
        got = rgb_planes(node.vszip.ColorMap(color=k).get_frame(0))
        assert_same_planes(got, colormap(src["planes"][0], bits, k), f"{fmt} noise color={k}")


def test_yuv_output_ignores_chroma():
    a = noise_clip("YUV420P8", 258, 130, seed=7)
    b = {"format": "YUV420P8", "planes": [a["planes"][0], 255 - a["planes"][1], a["planes"][2] // 3]}
    got_a = rgb_planes(to_node(a).vszip.ColorMap(13).get_frame(0))
    got_b = rgb_planes(to_node(b).vszip.ColorMap(13).get_frame(0))
    assert_same_planes(got_a, got_b, "chroma changed")
    assert_same_planes(got_a, colormap(a["planes"][0], 8, 13), "YUV420P8 luma")


def test_props():
    node = vz.core.clip_from_frames("GRAY16", [noise_clip("GRAY16", 64, 36, seed=1)["planes"]], props={"_ColorRange": 1, "_Matrix": 1, "x": 3})
    fr = node.vszip.ColorMap().get_frame(0)
    assert fr.props == {"_ColorRange": 0, "_Matrix": 0, "x": 3}


def test_device_batch_equals_get_frame():
    fmt, w, h, n = "YUV420P10", 642, 362, 12
    a, d = vz.DeviceClip(fmt, w, h, n), vz.DeviceClip("RGB24", w, h, n)
    a.fill_noise(seed=9)
    frames = [a.download(i) for i in range(n)]
    node = vz.core.clip_from_frames(fmt, frames).vszip.ColorMap(4)
    vz.ColorMapFilter(a.info(), 4).run_device(a, d, first=3, count=7)
    vz.core.sync()
    for i in range(3, 10):
        assert_same_planes(d.download(i), node.get_frame(i).planes, f"frame {i}")
    with pytest.raises(vz.Error, match="^ColorMap: device clip does not match the format the filter was created for$"):
        vz.ColorMapFilter(a.info(), 4).run_device(a, a)


def test_4k_gray16_device_batch():
    w, h, n = 3840, 2160, 3
    a, d = vz.DeviceClip("GRAY16", w, h, n), vz.DeviceClip("RGB24", w, h, n)
    a.fill_noise(seed=77)
    vz.ColorMapFilter(a.info(), 20).run_device(a, d)
    vz.core.sync()
    for i in range(n):
        assert_same_planes(d.download(i), colormap(a.download(i)[0], 16, 20), f"4K GRAY16 frame {i}")


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


def test_boxblur_clahe_colormap_uploads_gray_and_downloads_rgb():
    src = fx.make_clip("GRAY8", "odd")
    y = src["planes"][0]
    fused, moved = _fused_and_plain(src, lambda c: c.vszip.BoxBlur(hradius=2, vradius=2).vszip.CLAHE(limit=3).vszip.ColorMap(2))
    assert moved == (y.nbytes, 3 * y.size)
    want = colormap(clahe_plane(oracle.boxblur_plane(y, 2, 1, 2, 1), 8, 3, (3, 3)), 8, 2)
    assert_same_planes(rgb_planes(fused), want, "BoxBlur -> CLAHE -> ColorMap")


@pytest.mark.parametrize("fmt", ["GRAY16", "YUV420P8"])
def test_colormap_boxblur_planeminmax_chain(fmt):
    src = noise_clip(fmt, 322, 182, seed=12)
    fused, _ = _fused_and_plain(src, lambda c: c.vszip.ColorMap(16).vszip.BoxBlur(hradius=3, vradius=1).vszip.PlaneMinMax(planes=[0, 1, 2]))
    bits = vz.FORMATS[fmt].bits_per_sample
    want = [oracle.boxblur_plane(p, 3, 1, 1, 1) for p in colormap(src["planes"][0], bits, 16)]
    assert_same_planes(rgb_planes(fused), want, f"{fmt} ColorMap -> BoxBlur")
    assert fused.props["psmMin"] == [int(p.min()) for p in want] and fused.props["psmMax"] == [int(p.max()) for p in want]


def test_one_handle_many_threads():
    fmt, frames = "GRAY16", 24
    clips = [noise_clip(fmt, 322, 182, seed=900 + i) for i in range(frames)]
    want = [colormap(c["planes"][0], 16, 7) for c in clips]
    node = vz.core.clip_from_frames(fmt, [c["planes"] for c in clips]).vszip.ColorMap(7)
    order = [(i * 7) % frames for i in range(frames * 3)]
    with ThreadPoolExecutor(16) as ex:
        results = list(ex.map(lambda n: (n, node.get_frame(n)), order))
    for n, fr in results:
        assert_same_planes(rgb_planes(fr), want[n], f"ColorMap frame {n}")
