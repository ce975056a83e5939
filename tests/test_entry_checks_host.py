"""CPU-only: the exact message of every check an entry point makes before it touches a GPU (filters are created without a
device).  get_frame names missing or unexpected inputs as frames, the batched _device entry points as clips."""
import ctypes as C

import numpy as np
import pytest

import vapoursynth_zip_b200 as vz

W, H = 64, 48
NO_INIT = "vszip_cuda_init has not been called (no GPU context; there is no CPU fallback)"
BAD_CLIP = "device clip does not match the format the filter was created for"


@pytest.fixture(scope="module")
def lib():
    return vz.load_library()


@pytest.fixture(scope="module")
def flt():
    """GRAY8 instances of every filter, with and without their optional inputs."""
    vi = vz._vi(vz.GRAY8, W, H, 10)
    return {
        "BoxBlur": vz.BoxBlurFilter(vi),
        "Bilateral": vz.BilateralFilter(vi, None, sigmaS=2), "Bilateral+ref": vz.BilateralFilter(vi, vi, sigmaS=2),
        "PlaneMinMax": vz.PlaneMinMaxFilter(vi, None), "PlaneMinMax+clipb": vz.PlaneMinMaxFilter(vi, vi),
        "PlaneAverage": vz.PlaneAverageFilter(vi, None, exclude=[0]), "PlaneAverage+clipb": vz.PlaneAverageFilter(vi, vi, exclude=[0]),
        "Limiter": vz.LimiterFilter(vi),
        "LimitFilter": vz.LimitFilterFilter(vi, vi, None), "LimitFilter+ref": vz.LimitFilterFilter(vi, vi, vi),
        "AdaptiveBinarize": vz.AdaptiveBinarizeFilter(vi, vi),
    }


def _frame():
    return C.byref(vz._cframe([np.zeros((H, W), np.uint8)]))


# A zeroed struct where a device clip is expected: present, but of no format a filter is created for.
_FAKE = C.create_string_buffer(4096)
FAKE = C.addressof(_FAKE)


def _expect(msg, rc):
    assert rc != 0
    assert vz._last_error() == msg


def _get_frame(lib, name, h, a=True, b=None, c=None, dst=True):
    """The get_frame of `name` with frames a (main), b (second input), c (third input) and dst; True = a frame, None = NULL."""
    fr = lambda x: _frame() if x else None
    if name in ("BoxBlur", "Limiter"):
        return getattr(lib, f"vszip_{name.lower()}_get_frame")(h, 0, fr(a), fr(dst))
    if name == "Bilateral":
        return lib.vszip_bilateral_get_frame(h, 0, fr(a), fr(b), fr(dst))
    if name == "PlaneMinMax":
        return lib.vszip_planeminmax_get_frame(h, 0, fr(a), fr(b), C.byref(vz._MinMaxProps()))
    if name == "PlaneAverage":
        return lib.vszip_planeaverage_get_frame(h, 0, fr(a), fr(b), C.byref(vz._AverageProps()))
    if name == "LimitFilter":
        return lib.vszip_limitfilter_get_frame(h, 0, fr(a), fr(b), fr(c), fr(dst))
    return lib.vszip_adaptivebinarize_get_frame(h, 0, fr(a), fr(b), fr(dst))


def _device(lib, name, h, a=FAKE, b=None, c=None, dst=FAKE):
    """The _device entry of `name` with clips a (main), b (second input), c (third input) and dst."""
    if name in ("BoxBlur", "Limiter"):
        return getattr(lib, f"vszip_{name.lower()}_device")(h, a, dst, 0, 1, None)
    if name == "Bilateral":
        return lib.vszip_bilateral_device(h, a, b, dst, 0, 1, None)
    if name == "PlaneMinMax":
        return lib.vszip_planeminmax_device(h, a, b, 0, 1, None, None)
    if name == "PlaneAverage":
        return lib.vszip_planeaverage_device(h, a, b, 0, 1, None, None)
    if name == "LimitFilter":
        return lib.vszip_limitfilter_device(h, a, b, c, dst, 0, 1, None)
    return lib.vszip_adaptivebinarize_device(h, a, b, dst, 0, 1, None)


KINDS = ["BoxBlur", "Bilateral", "PlaneMinMax", "PlaneAverage", "Limiter", "LimitFilter", "AdaptiveBinarize"]
# inputs each kind is always called with: LimitFilter's src, AdaptiveBinarize's clip2
REQUIRED = {"LimitFilter": dict(b=True), "AdaptiveBinarize": dict(b=True)}


@pytest.mark.parametrize("name", KINDS)
def test_bad_handle(lib, flt, name):
    other = flt["Limiter" if name != "Limiter" else "BoxBlur"].handle
    for h in (None, other):
        _expect(f"{name}: bad filter handle", _get_frame(lib, name, h, **REQUIRED.get(name, {})))
        dev = {k: FAKE for k in REQUIRED.get(name, {})}
        _expect(f"{name}: bad filter handle", _device(lib, name, h, **dev))


@pytest.mark.parametrize(("name", "slot", "word"), [
    ("Bilateral", "b", "ref"), ("PlaneMinMax", "b", "clipb"), ("PlaneAverage", "b", "clipb"), ("LimitFilter", "c", "ref"),
])
def test_optional_input_presence(lib, flt, name, slot, word):
    extra = REQUIRED.get(name, {})
    with_input = flt[f"{name}+{word}"].handle
    without = flt[name].handle
    frame_msg = f"{name}: {word} frame presence does not match the filter instance"
    clip_msg = f"{name}: {word}{'' if word == 'clipb' else ' clip'} presence does not match the filter instance"
    _expect(frame_msg, _get_frame(lib, name, without, **extra, **{slot: True}))
    _expect(frame_msg, _get_frame(lib, name, with_input, **extra))
    dev = {k: FAKE for k in extra}
    _expect(clip_msg, _device(lib, name, without, **dev, **{slot: FAKE}))
    _expect(clip_msg, _device(lib, name, with_input, **dev))


@pytest.mark.parametrize("missing", ["a", "b", "dst"])
def test_required_frames(lib, flt, missing):
    args = dict(a=True, b=True, dst=True)
    args[missing] = None
    _expect("LimitFilter: flt, src and dst frames are required", _get_frame(lib, "LimitFilter", flt["LimitFilter"].handle, **args))
    _expect("AdaptiveBinarize: clip, clip2 and dst frames are required",
            _get_frame(lib, "AdaptiveBinarize", flt["AdaptiveBinarize"].handle, **args))


@pytest.mark.parametrize(("name", "instance", "required", "optional"), [
    ("BoxBlur", "BoxBlur", "a dst", ""),
    ("Bilateral", "Bilateral", "a dst", ""), ("Bilateral", "Bilateral+ref", "a dst", "b"),
    ("PlaneMinMax", "PlaneMinMax", "a", ""), ("PlaneMinMax", "PlaneMinMax+clipb", "a", "b"),
    ("PlaneAverage", "PlaneAverage", "a", ""), ("PlaneAverage", "PlaneAverage+clipb", "a", "b"),
    ("Limiter", "Limiter", "a dst", ""),
    ("LimitFilter", "LimitFilter", "a b dst", ""), ("LimitFilter", "LimitFilter+ref", "a b dst", "c"),
    ("AdaptiveBinarize", "AdaptiveBinarize", "a b dst", ""),
])
def test_device_clip_format(lib, flt, name, instance, required, optional):
    """Each clip a _device call cannot do without, NULL (the others present but of no matching format), and all of them present."""
    clips = (required + " " + optional).split()
    for missing in required.split() + [None]:
        args = {k: (None if k == missing else FAKE) for k in clips}
        args.setdefault("dst", None)
        _expect(f"{name}: {BAD_CLIP}", _device(lib, name, flt[instance].handle, **args))


def test_planestats_device(lib, flt):
    mm, av, mmb, avb = (flt[k].handle for k in ("PlaneMinMax", "PlaneAverage", "PlaneMinMax+clipb", "PlaneAverage+clipb"))
    one = lambda m, a, clip: lib.vszip_planestats_device(m, a, clip, 0, 1, None, None, None, None)
    two = lambda m, a, clip, b: lib.vszip_planestats_device_b(m, a, clip, b, 0, 1, None, None, None, None)
    handles = "PlaneStats: a PlaneMinMax and a PlaneAverage handle are required"
    for m, a in [(av, mm), (None, av), (mm, None), (flt["BoxBlur"].handle, av)]:
        _expect(handles, one(m, a, FAKE))
        _expect(handles, two(m, a, FAKE, None))
    _expect("PlaneStats: filters created with clipb cannot be combined", one(mmb, av, FAKE))
    _expect("PlaneStats: filters created with clipb cannot be combined", one(mm, avb, FAKE))
    presence = "PlaneStats: clipb presence does not match the filter instances"
    _expect(presence, two(mm, av, FAKE, FAKE))
    _expect(presence, two(mmb, avb, FAKE, None))
    _expect(presence, two(mmb, av, FAKE, None))
    for bad in (None, FAKE):
        _expect(f"PlaneStats: {BAD_CLIP}", one(mm, av, bad))
        _expect(f"PlaneStats: {BAD_CLIP}", two(mm, av, bad, None))
        _expect(f"PlaneStats: {BAD_CLIP}", two(mmb, avb, bad, FAKE))
        _expect(f"PlaneStats: {BAD_CLIP}", two(mmb, av, bad, FAKE))


def _chain(lib, filters):
    h = lib.vszip_chain_create((C.c_void_p * len(filters))(*[f.handle for f in filters]), len(filters))
    assert h, vz._last_error()
    return h


def test_chain_get_frame(lib, flt):
    _expect("chain: bad handle", lib.vszip_chain_get_frame(None, 0, _frame(), _frame(), None))
    h = _chain(lib, [flt["BoxBlur"], flt["PlaneMinMax"]])
    try:
        _expect("chain: dst is required when the chain holds a pixel filter", lib.vszip_chain_get_frame(h, 0, _frame(), None, None))
    finally:
        lib.vszip_chain_free(h)


def test_uninitialised_route(lib, flt):
    """Valid calls on a library that vszip_cuda_init has not set up."""
    if lib.vszip_cuda_device_count() != 0:
        pytest.skip("the library was initialised in this process")
    for name in KINDS:
        _expect(f"{name}: {NO_INIT}", _get_frame(lib, name, flt[name].handle, **REQUIRED.get(name, {})))
    for name, slot, word in [("Bilateral", "b", "ref"), ("PlaneMinMax", "b", "clipb"), ("PlaneAverage", "b", "clipb"), ("LimitFilter", "c", "ref")]:
        extra = REQUIRED.get(name, {})
        _expect(f"{name}: {NO_INIT}", _get_frame(lib, name, flt[f"{name}+{word}"].handle, **extra, **{slot: True}))
    for filters, dst in [([flt["BoxBlur"], flt["PlaneMinMax"]], _frame()), ([flt["PlaneMinMax"]], None)]:
        h = _chain(lib, filters)
        try:
            _expect(f"chain: {NO_INIT}", lib.vszip_chain_get_frame(h, 0, _frame(), dst, None))
        finally:
            lib.vszip_chain_free(h)
