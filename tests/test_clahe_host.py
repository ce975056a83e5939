"""CPU-only checks of CLAHE: the reference restatement (clahe_ref.py) against OpenCV's cv2.createCLAHE(...).apply bit for
bit, a known answer for every depth that needs no OpenCV, the create-time messages of the C ABI and the namespace binding."""
import ctypes as C

import numpy as np
import pytest

import vapoursynth_zip_b200 as vz
from clahe_ref import clahe_plane
from oracle import fixtures as fx
from test_node_model_host import Recorder

LIMITS = [0.0, 1.0, 15.0, 40.0, 1000.0]
TILES = [(1, 1), (3, 3), (8, 8), (4, 2), (16, 5)]


def _cv2():
    return pytest.importorskip("cv2")


@pytest.mark.parametrize("geo", ["full", "odd", "tiny"])
@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY16", "YUV420P8", "YUV420P16"])
def test_reference_matches_opencv_on_the_fixture(fmt, geo):
    cv2 = _cv2()
    bits = fx.FORMATS[fmt][2]
    for plane in fx.make_clip(fmt, geo)["planes"]:
        for limit in LIMITS:
            for tiles in TILES:
                want = cv2.createCLAHE(limit, tiles).apply(plane)
                assert np.array_equal(clahe_plane(plane, bits, limit, tiles), want), (fmt, geo, plane.shape, limit, tiles)


@pytest.mark.parametrize(("h", "w"), [(48, 64), (47, 63), (7, 13), (1, 9), (9, 1), (540, 960)])
@pytest.mark.parametrize("bits", [8, 16])
def test_reference_matches_opencv_on_noise(bits, h, w):
    cv2 = _cv2()
    rng = np.random.default_rng(bits * 1000 + h + w)
    img = rng.integers(0, 1 << bits, (h, w)).astype(np.uint8 if bits == 8 else np.uint16)
    for limit in LIMITS:
        for tiles in TILES:
            want = cv2.createCLAHE(limit, tiles).apply(img)
            assert np.array_equal(clahe_plane(img, bits, limit, tiles), want), (bits, h, w, limit, tiles)


@pytest.mark.parametrize("bits", [8, 10, 12, 16])
def test_one_tile_without_limit_is_histogram_equalisation(bits):
    """tiles [1, 1], limit 0: every output is rint_even(f32(cdf[s]) * f32((2^bits - 1) / N))."""
    hs = 1 << bits
    rng = np.random.default_rng(bits)
    img = rng.integers(0, hs, (37, 53)).astype(np.uint8 if bits == 8 else np.uint16)
    cdf = np.cumsum(np.bincount(img.ravel(), minlength=hs))
    lut = np.clip(np.rint(cdf.astype(np.float32) * (np.float32(hs - 1) / np.float32(img.size))), 0, hs - 1)
    assert np.array_equal(clahe_plane(img, bits, 0, (1, 1)), lut[img].astype(img.dtype))


def test_out_of_range_samples_count_as_the_top_bin():
    rng = np.random.default_rng(11)
    img = rng.integers(0, 1024, (40, 70)).astype(np.uint16)
    wild = img.copy()
    wild[::3, ::5] = rng.integers(1024, 65536, wild[::3, ::5].shape)
    for limit, tiles in ((0, (1, 1)), (15, (3, 3)), (2, (4, 2))):
        want = clahe_plane(np.minimum(wild, 1023), 10, limit, tiles)
        got = clahe_plane(wild, 10, limit, tiles)
        assert np.array_equal(got, want), (limit, tiles)
        assert int(got.max()) <= 1023


# --------------------------------------------------------------------------- create-time messages, through the C ABI
def _create(fmt, limit=None, tiles=None):
    lib = vz.load_library()
    vi = vz._vi(vz.FORMATS[fmt], 64, 48, 1)
    t, nt = (None, 0) if tiles is None else vz._i64(tiles)
    h = lib.vszip_clahe_create(C.byref(vi), C.byref(vz._ClaheArgs(limit is not None, float(limit or 0), t, nt)))
    if h:
        lib.vszip_filter_free(h)
        return None
    return vz._last_error()


@pytest.mark.parametrize(("fmt", "limit", "tiles", "msg"), [
    ("GRAYS", None, None, "CLAHE: only 8-16 bit int formats supported."),
    ("GRAYH", None, None, "CLAHE: only 8-16 bit int formats supported."),
    ("GRAY32", None, None, "CLAHE: only 8-16 bit int formats supported."),
    ("YUV420PS", None, None, "CLAHE: only 8-16 bit int formats supported."),
    ("GRAY16", -1.0, None, "CLAHE: limit must be non-negative."),
    ("GRAY16", float("nan"), None, "CLAHE: limit must be non-negative."),
    ("GRAY8", None, [3, 3, 3], "CLAHE: tiles has too many elements (got 3, max 2)."),
    ("GRAY8", None, [0], "CLAHE: tiles values must be at least 1."),
    ("GRAY8", None, [4, -1], "CLAHE: tiles values must be at least 1."),
    ("GRAY8", None, [17], "CLAHE: at most 256 tiles per plane (tiles[0] * tiles[1])."),
    ("GRAY8", None, [257, 1], "CLAHE: at most 256 tiles per plane (tiles[0] * tiles[1])."),
    ("GRAY8", None, [1 << 40, 1 << 40], "CLAHE: at most 256 tiles per plane (tiles[0] * tiles[1])."),
    ("GRAY8", None, None, None), ("GRAY10", 0, [16], None), ("YUV420P16", 1e9, [256, 1], None), ("RGB48", 2.5, [1, 256], None),
])
def test_create_messages(fmt, limit, tiles, msg):
    assert _create(fmt, limit, tiles) == msg


# --------------------------------------------------------------------------- the namespace call
class ClaheRecorder(Recorder):
    """Also records the arguments vszip_clahe_create receives."""

    def __getattr__(self, name):
        if name == "vszip_clahe_create":
            real = getattr(self.real, name)

            def create(vi, args):
                a = args._obj
                self.calls.append(("create", a.has_limit, a.limit, [a.tiles[i] for i in range(a.num_tiles)]))
                return self._created("clahe", real(vi, args))
            return create
        return super().__getattr__(name)


@pytest.fixture
def crec():
    r = ClaheRecorder(vz.load_library())
    saved = vz._lib, vz.core._ready, vz.core.fuse_chains
    vz._lib, vz.core._ready, vz.core.fuse_chains = r, False, True
    try:
        yield r
    finally:
        vz._lib, vz.core._ready, vz.core.fuse_chains = saved


@pytest.mark.parametrize(("build", "args"), [
    (lambda a, core: a.vszip.CLAHE(), (0, 0.0, [])),
    (lambda a, core: core.vszip.CLAHE(a), (0, 0.0, [])),
    (lambda a, core: a.vszip.CLAHE(2.5, [4, 2]), (1, 2.5, [4, 2])),
    (lambda a, core: core.vszip.CLAHE(a, 0, 8), (1, 0.0, [8])),
    (lambda a, core: a.vszip.CLAHE(tiles=[16, 5], limit=40), (1, 40.0, [16, 5])),
    (lambda a, core: core.vszip.CLAHE(clip=a, limit=1), (1, 1.0, [])),
])
def test_namespace_binds_the_arguments(crec, build, args):
    a = crec.source("a", "YUV420P16", props={"_ColorRange": 1})
    node = build(a, vz.core)
    frame = node.get_frame(2)
    assert crec.calls == [("create",) + args, ("clahe", 2, [["a2.0", "a2.1", "a2.2"]], ["dst", "dst", "dst"])]
    assert crec.planes(frame) == ["dst", "dst", "dst"]
    assert frame.props == {"_ColorRange": 1, "tag": "a"}


def test_chains_through_clahe_are_fused(crec):
    a = crec.source("a", "GRAY16")
    node = a.vszip.BoxBlur(hradius=2, vradius=2).vszip.CLAHE(limit=3).vszip.PlaneMinMax()
    frame = node.get_frame(1)
    assert [c for c in crec.calls if c[0] != "create"] == [
        ("create2", ["boxblur", "clahe", "planeminmax"], [0, 1, 2], [-1, -1, -1], [-1, -1, -1]),
        ("chain", 1, ["a1.0", None, None], ["dst", None, None]),
    ]
    assert crec.planes(frame) == ["dst"] and frame.props["psmMin"] == 10
    crec.calls = []
    lf = a.vszip.CLAHE().vszip.LimitFilter(a, dark_thr=4)
    lf.get_frame(3)
    assert [c for c in crec.calls if c[0] != "create"] == [
        ("clahe", 0, [["a0.0", None, None]], ["dst", None, None]),  # LimitFilter reads _ColorRange from frame 0 of flt
        ("create2", ["clahe", "limitfilter"], [0, 1], [-1, 0], [-1, -1]),
        ("chain", 3, ["a3.0", None, None], ["dst", None, None]),
    ]
