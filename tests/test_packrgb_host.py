"""CPU-only checks of PackRGB: the create-time message of the C ABI, the output format and read planes it reports, the Python node
(format, binding, planes, props) and the chains it may join, including the planes a chain ending in it writes."""
import ctypes as C

import numpy as np
import pytest

import vapoursynth_zip_b200 as vz
from test_node_model_host import Recorder

W, H = 64, 32  # the size of Recorder.source clips
MSG = "PackRGB: only RGB24 and RGB30 clips are supported."


def _vi(fmt, w=W, h=H):
    return vz._vi(vz.FORMATS[fmt], w, h, 10)


def _create(vi):
    lib = vz.load_library()
    h = lib.vszip_packrgb_create(C.byref(vi))
    if h:
        lib.vszip_filter_free(h)
        return None
    return vz._last_error()


@pytest.mark.parametrize(("fmt", "msg"), [
    ("GRAY8", MSG), ("GRAY32", MSG), ("YUV444P8", MSG), ("YUV444P10", MSG), ("RGB48", MSG), ("RGBH", MSG), ("RGBS", MSG),
    ("RGB24", None), ("RGB30", None),
])
def test_create_messages(fmt, msg):
    assert _create(_vi(fmt)) == msg


def test_create_rejects_other_rgb_depths():
    rgb9 = vz._VideoInfo(W, H, 10, vz.RGB, vz.INTEGER, 9, 2, 0, 0, 3)
    assert _create(rgb9) == MSG
    rgb30_in_bytes = vz._VideoInfo(W, H, 10, vz.RGB, vz.INTEGER, 10, 1, 0, 0, 3)
    assert _create(rgb30_in_bytes) == MSG
    assert _create(vz._VideoInfo(0, H, 10, vz.RGB, vz.INTEGER, 8, 1, 0, 0, 3)) == "PackRGB: invalid video info"


def _out_info(f):
    o = vz._VideoInfo()
    vz._check(vz.load_library().vszip_filter_output_info(f.handle, C.byref(o)))
    return (o.width, o.height, o.num_frames, o.color_family, o.sample_type, o.bits_per_sample, o.bytes_per_sample, o.sub_sampling_w,
            o.sub_sampling_h, o.num_planes)


@pytest.mark.parametrize("fmt", ["RGB24", "RGB30"])
def test_output_info_and_read_planes(fmt):
    f = vz.PackRGBFilter(_vi(fmt, 70, 30))
    assert _out_info(f) == (70, 30, 10, vz.GRAY, vz.INTEGER, 32, 4, 0, 0, 1)
    assert f.process == [True, True, True]


# --------------------------------------------------------------------------- the Python node
@pytest.fixture
def rec():
    r = Recorder(vz.load_library())
    saved = vz._lib, vz.core._ready, vz.core.fuse_chains
    vz._lib, vz.core._ready, vz.core.fuse_chains = r, False, True
    try:
        yield r
    finally:
        vz._lib, vz.core._ready, vz.core.fuse_chains = saved


@pytest.mark.parametrize("fmt", ["RGB24", "RGB30"])
@pytest.mark.parametrize("build", [lambda a, core: a.vszip.PackRGB(), lambda a, core: core.vszip.PackRGB(a),
                                   lambda a, core: core.vszip.PackRGB(clip=a)])
def test_node_format_binding_and_props(rec, fmt, build):
    a = rec.source("a", fmt, props={"_ColorRange": 0, "_Matrix": 0})
    node = build(a, vz.core)
    assert node.format is vz.GRAY32 and (node.width, node.height, node.num_frames) == (W, H, 4)
    frame = node.get_frame(2)
    assert rec.calls == [("packrgb", 2, [["a2.0", "a2.1", "a2.2"]], ["dst", None, None])]  # reads three planes, writes one
    assert frame.format is vz.GRAY32 and [(p.shape, p.dtype) for p in frame.planes] == [((H, W), np.uint32)]
    assert rec.planes(frame) == ["dst"]
    assert frame.props == {"_ColorRange": 0, "_Matrix": 0, "tag": "a"}


def test_node_binding_errors():
    a = vz.core.BlankClip("RGB24", W, H)
    with pytest.raises(vz.Error, match="^too many positional arguments$"):
        a.vszip.PackRGB(1)
    with pytest.raises(vz.Error, match="^clip argument is required$"):
        vz.core.vszip.PackRGB()
    with pytest.raises(vz.Error, match=f"^{MSG}$"):
        vz.core.BlankClip("GRAY8", W, H).vszip.PackRGB()


def test_fused_chain_returns_gray32(rec):
    a = rec.source("a", "GRAY8", props={"_ColorRange": 1})
    node = a.vszip.BoxBlur(hradius=2, vradius=2).vszip.CLAHE(limit=3).vszip.ColorMap(2).vszip.PackRGB()
    assert node.format is vz.GRAY32
    frame = node.get_frame(1)
    assert rec.calls == [
        ("create2", ["boxblur", "clahe", "colormap", "packrgb"], [0, 1, 2, 3], [-1] * 4, [-1] * 4),
        ("chain", 1, ["a1.0", None, None], ["dst", None, None]),
    ]
    assert frame.format is vz.GRAY32 and [(p.shape, p.dtype) for p in frame.planes] == [((H, W), np.uint32)]
    assert frame.props == {"_ColorRange": 0, "_Matrix": 0, "tag": "a"}  # ColorMap's props, passed on unchanged


# --------------------------------------------------------------------------- chains through the C ABI
def _chain(filters, inputs=None, linear=False):
    lib, n = vz.load_library(), len(filters)
    handles = (C.c_void_p * n)(*[f.handle for f in filters])
    arr = lambda v: None if v is None else (C.c_int32 * n)(*v)
    h = lib.vszip_chain_create(handles, n) if linear else lib.vszip_chain_create2(handles, n, arr(inputs), None, None)
    if not h:
        raise vz.Error(vz._last_error())
    w = (C.c_int32 * 3)()
    lib.vszip_chain_planes(h, C.byref(w))
    lib.vszip_chain_free(h)
    return list(w)


@pytest.mark.parametrize("linear", [True, False])
def test_chains_into_packrgb_are_accepted(linear):
    gray, rgb24, rgb30 = _vi("GRAY8"), _vi("RGB24"), _vi("RGB30")
    assert _chain([vz.ColorMapFilter(gray), vz.PackRGBFilter(rgb24)], [0, 1], linear=linear) == [1, 0, 0]
    assert _chain([vz.BoxBlurFilter(rgb24), vz.PackRGBFilter(rgb24)], [0, 1], linear=linear) == [1, 0, 0]
    assert _chain([vz.LimiterFilter(rgb30, tv_range=True), vz.PackRGBFilter(rgb30)], [0, 1], linear=linear) == [1, 0, 0]
    assert _chain([vz.BoxBlurFilter(gray), vz.CLAHEFilter(gray), vz.ColorMapFilter(gray), vz.PackRGBFilter(rgb24)], [0, 1, 2, 3],
                  linear=linear) == [1, 0, 0]
    # a BoxBlur of one RGB plane still ends in the one packed plane
    assert _chain([vz.BoxBlurFilter(rgb24, planes=[2]), vz.PackRGBFilter(rgb24)], [0, 1], linear=linear) == [1, 0, 0]
    # statistics of the source next to a PackRGB of it
    assert _chain([vz.PackRGBFilter(rgb24), vz.PlaneMinMaxFilter(rgb24)], [0, 0]) == [0, 0, 0]


@pytest.mark.parametrize("linear", [True, False])
def test_chains_reading_the_wrong_format_are_rejected(linear):
    gray, rgb24 = _vi("GRAY8"), _vi("RGB24")
    with pytest.raises(vz.Error) as e:
        _chain([vz.BoxBlurFilter(gray), vz.PackRGBFilter(rgb24)], [0, 1], linear=linear)
    assert str(e.value) == "chain: filter 1 was created for a different video format than filter 0"
    with pytest.raises(vz.Error) as e:
        _chain([vz.PackRGBFilter(rgb24), vz.BoxBlurFilter(rgb24)], [0, 1], linear=linear)
    assert str(e.value) == "chain: filter 1 was created for a different video format than the value it reads"
    with pytest.raises(vz.Error) as e:
        _chain([vz.ColorMapFilter(gray), vz.PackRGBFilter(rgb24), vz.PackRGBFilter(rgb24)], [0, 1, 2], linear=linear)
    assert str(e.value) == "chain: filter 2 was created for a different video format than the value it reads"
