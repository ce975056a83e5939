"""CPU-only checks of ColorMap: the create-time messages and the default of the C ABI, the tables against OpenCV, the output format
every filter reports, the Python node (format, binding, props, output planes) and the chains a format-changing filter may join."""
import ctypes as C

import numpy as np
import pytest

import vapoursynth_zip_b200 as vz
from test_node_model_host import Recorder

W, H = 64, 32  # the size of Recorder.source clips


def _vi(fmt, w=W, h=H):
    return vz._vi(vz.FORMATS[fmt], w, h, 10)


def _create(fmt, color=None):
    lib = vz.load_library()
    h = lib.vszip_colormap_create(C.byref(_vi(fmt)), C.byref(vz._ColorMapArgs(color is not None, int(color or 0))))
    if h:
        lib.vszip_filter_free(h)
        return None
    return vz._last_error()


@pytest.mark.parametrize(("fmt", "color", "msg"), [
    ("GRAYS", None, "ColorMap: only 8-16 bit int formats supported."),
    ("GRAYH", None, "ColorMap: only 8-16 bit int formats supported."),
    ("GRAY32", None, "ColorMap: only 8-16 bit int formats supported."),
    ("YUV420PS", None, "ColorMap: only 8-16 bit int formats supported."),
    ("RGBS", None, "ColorMap: only 8-16 bit int formats supported."),
    ("RGB24", None, "ColorMap: clip must be GRAY or YUV."),
    ("RGB48", 3, "ColorMap: clip must be GRAY or YUV."),
    ("GRAY8", -1, "ColorMap: color must be between 0 and 21."),
    ("GRAY8", 22, "ColorMap: color must be between 0 and 21."),
    ("YUV420P10", 1 << 40, "ColorMap: color must be between 0 and 21."),
    ("GRAY8", None, None), ("GRAY8", 0, None), ("GRAY16", 21, None), ("YUV420P10", 5, None), ("YUV444P16", 20, None),
])
def test_create_messages(fmt, color, msg):
    assert _create(fmt, color) == msg


def test_default_color_is_turbo():
    assert np.array_equal(vz.ColorMapFilter(_vi("GRAY8")).lut(), vz.ColorMapFilter(_vi("GRAY8"), 20).lut())
    assert not np.array_equal(vz.ColorMapFilter(_vi("GRAY8")).lut(), vz.ColorMapFilter(_vi("GRAY8"), 2).lut())


def test_tables_equal_opencv():
    cv2 = pytest.importorskip("cv2")
    ramp = np.arange(256, dtype=np.uint8)[:, None]
    for k in range(22):
        want = cv2.applyColorMap(ramp, k)[:, 0, ::-1]
        assert np.array_equal(vz.ColorMapFilter(_vi("GRAY16"), k).lut(), want), k


def _out_info(f):
    o = vz._VideoInfo()
    vz._check(vz.load_library().vszip_filter_output_info(f.handle, C.byref(o)))
    return (o.width, o.height, o.num_frames, o.color_family, o.sample_type, o.bits_per_sample, o.bytes_per_sample, o.sub_sampling_w,
            o.sub_sampling_h, o.num_planes)


def _info(vi):
    return (vi.width, vi.height, vi.num_frames, vi.color_family, vi.sample_type, vi.bits_per_sample, vi.bytes_per_sample,
            vi.sub_sampling_w, vi.sub_sampling_h, vi.num_planes)


@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY10", "YUV420P16"])
def test_output_info(fmt):
    vi = _vi(fmt, 70, 30)
    assert _out_info(vz.ColorMapFilter(vi)) == (70, 30, 10, vz.RGB, vz.INTEGER, 8, 1, 0, 0, 3)
    assert _out_info(vz.BoxBlurFilter(vi)) == _info(vi)
    assert _out_info(vz.CLAHEFilter(vi)) == _info(vi)
    assert _out_info(vz.PlaneMinMaxFilter(vi)) == _info(vi)
    planes = (C.c_int32 * 3)()
    vz.load_library().vszip_filter_planes(vz.ColorMapFilter(vi).handle, C.byref(planes))
    assert list(planes) == [1, 0, 0]  # the planes it reads


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


@pytest.mark.parametrize(("build", "color"), [
    (lambda a, core: a.vszip.ColorMap(), 20),
    (lambda a, core: core.vszip.ColorMap(a), 20),
    (lambda a, core: a.vszip.ColorMap(5), 5),
    (lambda a, core: core.vszip.ColorMap(a, 0), 0),
    (lambda a, core: a.vszip.ColorMap(color=21), 21),
    (lambda a, core: core.vszip.ColorMap(clip=a, color=11), 11),
])
def test_node_format_binding_and_props(rec, build, color):
    a = rec.source("a", "YUV420P10", props={"_ColorRange": 1, "_Matrix": 1})
    node = build(a, vz.core)
    assert node.format is vz.RGB24 and (node.width, node.height, node.num_frames) == (W, H, 4)
    assert np.array_equal(node.filter.lut(), vz.ColorMapFilter(_vi("GRAY8"), color).lut())
    frame = node.get_frame(2)
    assert rec.calls == [("colormap", 2, [["a2.0", None, None]], ["dst", "dst", "dst"])]  # reads the luma, writes three planes
    assert frame.format is vz.RGB24 and [(p.shape, p.dtype) for p in frame.planes] == [((H, W), np.uint8)] * 3
    assert rec.planes(frame) == ["dst", "dst", "dst"]
    assert frame.props == {"_ColorRange": 0, "_Matrix": 0, "tag": "a"}


def test_fused_chain_returns_rgb(rec):
    a = rec.source("a", "GRAY16")
    node = a.vszip.BoxBlur(hradius=2, vradius=2).vszip.CLAHE(limit=3).vszip.ColorMap(2)
    assert node.format is vz.RGB24
    frame = node.get_frame(1)
    assert rec.calls == [
        ("create2", ["boxblur", "clahe", "colormap"], [0, 1, 2], [-1, -1, -1], [-1, -1, -1]),
        ("chain", 1, ["a1.0", None, None], ["dst", "dst", "dst"]),
    ]
    assert frame.format is vz.RGB24 and [(p.shape, p.dtype) for p in frame.planes] == [((H, W), np.uint8)] * 3
    assert frame.props == {"_ColorRange": 0, "_Matrix": 0, "tag": "a"}
    rec.calls = []
    m = a.vszip.ColorMap().vszip.BoxBlur().vszip.PlaneMinMax()
    frame = m.get_frame(0)
    assert rec.calls[0] == ("create2", ["colormap", "boxblur", "planeminmax"], [0, 1, 2], [-1, -1, -1], [-1, -1, -1])
    assert frame.format is vz.RGB24 and rec.planes(frame) == ["dst", "dst", "dst"] and "psmMin" in frame.props


# --------------------------------------------------------------------------- chains through the C ABI
def _chain(filters, inputs=None, second=None, linear=False):
    lib, n = vz.load_library(), len(filters)
    handles = (C.c_void_p * n)(*[f.handle for f in filters])
    arr = lambda v: None if v is None else (C.c_int32 * n)(*v)
    h = lib.vszip_chain_create(handles, n) if linear else lib.vszip_chain_create2(handles, n, arr(inputs), arr(second), None)
    if not h:
        raise vz.Error(vz._last_error())
    w = (C.c_int32 * 3)()
    lib.vszip_chain_planes(h, C.byref(w))
    lib.vszip_chain_free(h)
    return list(w)


@pytest.mark.parametrize("linear", [True, False])
def test_chains_through_colormap_are_accepted(linear):
    gray, rgb = _vi("GRAY8"), _vi("RGB24")
    assert _chain([vz.CLAHEFilter(gray), vz.ColorMapFilter(gray)], [0, 1], linear=linear) == [1, 1, 1]
    assert _chain([vz.ColorMapFilter(gray), vz.BoxBlurFilter(rgb)], [0, 1], linear=linear) == [1, 1, 1]
    # a BoxBlur of one RGB plane still returns every plane: the others come from the ColorMap, not from the source
    assert _chain([vz.ColorMapFilter(gray), vz.BoxBlurFilter(rgb, planes=[1])], [0, 1], linear=linear) == [1, 1, 1]
    yuv = _vi("YUV420P16")
    assert _chain([vz.ColorMapFilter(yuv), vz.BoxBlurFilter(rgb), vz.PlaneMinMaxFilter(rgb)], [0, 1, 2], linear=linear) == [1, 1, 1]
    # statistics of the source next to a ColorMap of it
    assert _chain([vz.ColorMapFilter(gray), vz.PlaneMinMaxFilter(gray)], [0, 0]) == [0, 0, 0]


@pytest.mark.parametrize("linear", [True, False])
def test_chains_reading_the_wrong_format_are_rejected(linear):
    gray, rgb = _vi("GRAY8"), _vi("RGB24")
    with pytest.raises(vz.Error) as e:
        _chain([vz.ColorMapFilter(gray), vz.BoxBlurFilter(gray)], [0, 1], linear=linear)
    assert str(e.value) == "chain: filter 1 was created for a different video format than the value it reads"
    # a diamond LimitFilter after the ColorMap: flt is RGB24, src the GRAY8 source
    lf = vz.LimitFilterFilter(rgb, rgb, None, dark_thr=4)
    with pytest.raises(vz.Error) as e:
        _chain([vz.ColorMapFilter(gray), lf], [0, 1], [-1, 0], linear=linear)
    assert str(e.value) == "chain: filter 1 was created for a different video format than filter 0"
    # a filter created for RGB24 cannot read the gray source either
    with pytest.raises(vz.Error) as e:
        _chain([vz.ColorMapFilter(gray), vz.BoxBlurFilter(rgb), vz.BoxBlurFilter(rgb)], [0, 1, 0])
    assert str(e.value) == "chain: filter 2 was created for a different video format than filter 0"
