"""CLAHE on the GPU: bit-exact with clahe_ref.py (itself pinned against OpenCV by test_clahe_host.py) on every integer family, with
OpenCV directly, in device batches that span several L2 chunks, in fused chains and from 16 host threads on one handle."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
import vapoursynth_zip_b200 as vz
from clahe_ref import clahe_plane
from helpers import assert_same_planes, from_frame, noise_clip, to_node
from oracle import fixtures as fx

pytestmark = pytest.mark.gpu

# (limit, tiles): None = the default
CASES = [(None, None), (0, [1, 1]), (1, [3, 3]), (15, [8, 8]), (40, [4, 2]), (1000, [16, 5]), (2.5, [16, 5]), (15, [2]), (0, [8, 8])]


def clahe(clip, limit=None, tiles=None):
    bits = fx.FORMATS[clip["format"]][2]
    lim = 15.0 if limit is None else limit
    t = [3, 3] if tiles is None else (tiles * 2 if len(tiles) == 1 else tiles)
    return {"format": clip["format"], "planes": [clahe_plane(p, bits, lim, t) for p in clip["planes"]]}


def _args(limit, tiles):
    return {k: v for k, v in (("limit", limit), ("tiles", tiles)) if v is not None}


@pytest.mark.parametrize("geo", ["full", "odd", "tiny"])
@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY10", "GRAY16", "YUV420P8", "YUV420P10", "YUV420P16", "RGB24", "RGB48"])
def test_fixture_against_the_oracle(fmt, geo):
    src = fx.make_clip(fmt, geo)
    node = to_node(src)
    for limit, tiles in CASES:
        got = from_frame(fmt, node.vszip.CLAHE(**_args(limit, tiles)).get_frame(0))
        assert_same_planes(got["planes"], clahe(src, limit, tiles)["planes"], f"{fmt} {geo} limit={limit} tiles={tiles}")


@pytest.mark.parametrize(("fmt", "w", "h"), [("GRAY8", 517, 243), ("GRAY16", 517, 243), ("YUV420P10", 322, 182), ("RGB48", 130, 66)])
def test_noise_against_the_oracle(fmt, w, h):
    src = noise_clip(fmt, w, h, seed=41)
    node = to_node(src)
    for limit, tiles in CASES:
        got = from_frame(fmt, node.vszip.CLAHE(**_args(limit, tiles)).get_frame(0))
        assert_same_planes(got["planes"], clahe(src, limit, tiles)["planes"], f"{fmt} noise limit={limit} tiles={tiles}")


def test_out_of_range_10_bit_samples():
    """Samples above 1023 in a 10-bit clip count as 1023 (no LUT index leaves the table)."""
    src = noise_clip("GRAY16", 200, 120, seed=42)
    src = {"format": "GRAY10", "planes": [src["planes"][0] >> 5]}   # 0..2047
    got = from_frame("GRAY10", to_node(src).vszip.CLAHE(limit=2, tiles=[4, 2]).get_frame(0))
    assert_same_planes(got["planes"], clahe(src, 2, [4, 2])["planes"], "10-bit out of range")
    assert int(got["planes"][0].max()) <= 1023


@pytest.mark.parametrize(("fmt", "color"), [("YUV420P16", [0, 32768, 65535]), ("GRAY8", [77]), ("RGB24", [0, 128, 255])])
def test_constant_clip(fmt, color):
    node = vz.core.BlankClip(fmt, 640, 360, color=color)
    src = from_frame(fmt, node.get_frame(0))
    for limit, tiles in CASES[:4]:
        got = from_frame(fmt, node.vszip.CLAHE(**_args(limit, tiles)).get_frame(0))
        assert_same_planes(got["planes"], clahe(src, limit, tiles)["planes"], f"BlankClip {fmt} {color} limit={limit} tiles={tiles}")


@pytest.mark.parametrize("bits", [8, 16])
def test_planes_against_opencv(bits):
    cv2 = pytest.importorskip("cv2")
    fmt = "GRAY8" if bits == 8 else "GRAY16"
    for geo in ("full", "odd"):
        plane = fx.make_clip(fmt, geo)["planes"][0]
        for limit, tiles in ((15.0, (3, 3)), (2.0, (8, 8)), (0.0, (4, 2)), (40.0, (16, 5))):
            got = to_node({"format": fmt, "planes": [plane]}).vszip.CLAHE(limit=limit, tiles=list(tiles)).get_frame(0).planes[0]
            assert np.array_equal(got, cv2.createCLAHE(limit, tiles).apply(plane)), (fmt, geo, limit, tiles)


@pytest.mark.parametrize(("fmt", "w", "h", "tiles"), [("YUV420P16", 1920, 1080, [3, 3]), ("YUV420P16", 1920, 1080, [8, 8]),
                                                      ("GRAY16", 3840, 2160, [8, 8]), ("YUV420P8", 1920, 1080, [8, 8])])
def test_full_size_noise(fmt, w, h, tiles):
    a, d = vz.DeviceClip(fmt, w, h, 2), vz.DeviceClip(fmt, w, h, 2)
    a.fill_noise(seed=77)
    vz.CLAHEFilter(a.info(), limit=15, tiles=tiles).run_device(a, d)
    for i in range(2):
        want = clahe({"format": fmt, "planes": a.download(i)}, 15, tiles)
        assert_same_planes(d.download(i), want["planes"], f"{fmt} {w}x{h} tiles={tiles} frame {i}")


def test_device_batch_equals_get_frame():
    """first > 0 and enough frames for several L2 chunks (a YUV420P16 640x360 frame with 3x3 tiles needs ~12 MB of tables)."""
    fmt, w, h, n = "YUV420P16", 640, 360, 24
    a, d = vz.DeviceClip(fmt, w, h, n), vz.DeviceClip(fmt, w, h, n)
    a.fill_noise(seed=9)
    frames = [a.download(i) for i in range(n)]
    node = vz.core.clip_from_frames(fmt, frames).vszip.CLAHE(limit=4)
    vz.CLAHEFilter(a.info(), limit=4).run_device(a, d, first=3, count=19)
    for i in range(3, 22):
        assert_same_planes(d.download(i), node.get_frame(i).planes, f"frame {i}")


def _fused_vs_unfused(src, build):
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
    fb = sum(p.nbytes for p in src["planes"])
    assert (after[0] - before[0], after[1] - before[1]) == (fb, fb)
    assert_same_planes(fused.planes, plain.planes, "fused vs unfused")
    assert fused.props == plain.props, (fused.props, plain.props)
    return fused


@pytest.mark.parametrize("fmt", ["YUV420P16", "YUV420P8", "GRAY10"])
def test_boxblur_clahe_planeminmax_chain(fmt):
    src = fx.make_clip(fmt, "odd")
    fused = _fused_vs_unfused(src, lambda c: c.vszip.BoxBlur(hradius=2, vradius=2).vszip.CLAHE(limit=3).vszip.PlaneMinMax(planes=[0]))
    want = clahe(oracle_boxblur(src), 3)
    assert_same_planes(fused.planes, want["planes"], f"{fmt} BoxBlur -> CLAHE")


def oracle_boxblur(clip):
    return {"format": clip["format"], "planes": [oracle.boxblur_plane(p, 2, 1, 2, 1) for p in clip["planes"]]}


@pytest.mark.parametrize("fmt", ["YUV420P16", "RGB24"])
def test_clahe_limitfilter_chain(fmt):
    src = noise_clip(fmt, 322, 182, seed=12)
    _fused_vs_unfused(src, lambda c: c.vszip.CLAHE(tiles=[4, 2]).vszip.LimitFilter(c, dark_thr=8, bright_thr=4, elast=3))


def test_one_handle_many_threads():
    fmt, frames = "YUV420P16", 24
    clips = [noise_clip(fmt, 322, 182, seed=900 + i) for i in range(frames)]
    want = [clahe(c, 2, [4, 2])["planes"] for c in clips]
    node = vz.core.clip_from_frames(fmt, [c["planes"] for c in clips]).vszip.CLAHE(limit=2, tiles=[4, 2])
    order = [(i * 7) % frames for i in range(frames * 3)]
    with ThreadPoolExecutor(16) as ex:
        results = list(ex.map(lambda n: (n, node.get_frame(n)), order))
    for n, fr in results:
        assert_same_planes(fr.planes, want[n], f"CLAHE frame {n}")
