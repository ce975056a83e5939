"""Fused chains that are small DAGs (vszip_chain_create2): clipb / ref / src inputs taken from the chain's source or from an earlier
element, evaluated with one upload and one download, identical to the unfused nodes and to the oracle.  Also the one-read
PlaneMinMax + PlaneAverage with clipb (vszip_planestats_device_b)."""
import numpy as np
import pytest

import oracle_api as oa
import vapoursynth_zip_b200 as vz
from helpers import assert_same_planes, noise_clip, to_node

pytestmark = pytest.mark.gpu


def _frame_bytes(clip):
    return sum(p.nbytes for p in clip["planes"])


def _dag_case(clip, build, down=True):
    """Fused vs VSZIP_FUSE_CHAINS=0: same planes, same props; the fused frame moved one frame up and one (or no) frame down."""
    vz.core.fuse_chains = True
    try:
        node = build(to_node(clip))
        before = vz.core.transfer_bytes()
        fused = node.get_frame(0)
        after = vz.core.transfer_bytes()
        assert getattr(node, "_chain", None) is not None, "the chain was not fused"
    finally:
        vz.core.fuse_chains = False
    try:
        plain = build(to_node(clip)).get_frame(0)
    finally:
        vz.core.fuse_chains = True
    fb = _frame_bytes(clip)
    assert (after[0] - before[0], after[1] - before[1]) == (fb, fb if down else 0)
    assert_same_planes(fused.planes, plain.planes, "fused vs unfused")
    assert fused.props == plain.props, (fused.props, plain.props)
    return node, fused


def _planes(frame):
    return [np.ascontiguousarray(p) for p in frame.planes]


def _close(got, want, what, exact=False):
    for i, (g, w) in enumerate(zip(got, want)):
        if exact or g.dtype.kind != "f":
            if exact:
                assert_same_planes([g], [w], f"{what} plane {i}")
            else:
                assert np.abs(g.astype(np.int64) - w.astype(np.int64)).max() <= 1, f"{what} plane {i}"
        else:
            g64, w64 = g.astype(np.float64), w.astype(np.float64)
            rel = 1e-5 if g.dtype == np.float32 else 1e-3
            assert (np.abs(g64 - w64) <= rel * np.abs(w64) + 1e-6).all(), f"{what} plane {i}"


def _props_match(got, want):
    for k, w in want.items():
        g = got[k]
        for a, b in zip(g if isinstance(g, list) else [g], w if isinstance(w, list) else [w]):
            assert a == b if isinstance(b, int) else a == pytest.approx(b, rel=1e-12, abs=1e-300), (k, got, want)


@pytest.mark.parametrize("thr", [None, 0.1])
@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY16", "GRAYH", "GRAYS"])
@pytest.mark.parametrize(("w", "h"), [(322, 182), (640, 96)])
def test_boxblur_then_minmax_against_the_source(fmt, w, h, thr):
    clip = noise_clip(fmt, w, h, seed=5)
    kw = {} if thr is None else dict(minthr=thr, maxthr=thr)
    node, f = _dag_case(clip, lambda c: c.vszip.BoxBlur(hradius=2, vradius=2).vszip.PlaneMinMax(clipb=c, **kw))
    want = oa.boxblur(clip, hradius=2, vradius=2)
    assert_same_planes(f.planes, want["planes"], "BoxBlur")
    _props_match(f.props, oa.planeminmax(want, clipb=clip, **kw))
    assert len(node._chain[0].nodes) == 2


@pytest.mark.parametrize(("w", "h"), [(322, 182), (640, 360)])
def test_minmax_and_average_pair_with_clipb(w, h):
    """psmDiff: how much the blur changed the frame, PlaneMinMax + PlaneAverage of the same pair (one read when fused)."""
    clip = noise_clip("YUV420P16", w, h, seed=6)

    def build(c):
        m = c.vszip.BoxBlur(hradius=2, vradius=2).vszip.PlaneMinMax(minthr=0.1, maxthr=0.1, clipb=c, planes=[0, 1, 2])
        return m.vszip.PlaneAverage(exclude=[0], clipb=c, planes=[0, 1, 2], prop="a")
    _, f = _dag_case(clip, build)
    blur = oa.boxblur(clip, hradius=2, vradius=2)
    want = oa.planeminmax(blur, minthr=0.1, maxthr=0.1, clipb=clip, planes=[0, 1, 2])
    want.update(oa.planeaverage(blur, [0], clipb=clip, planes=[0, 1, 2], prop="a"))
    _props_match(f.props, want)
    assert f.props["psmDiff"] == f.props["aDiff"]


@pytest.mark.parametrize("fmt", ["GRAYS", "GRAYH"])
def test_float_pair_with_clipb_and_thresholds(fmt):
    """Rows without padding (640 * 4 bytes) are not fused with thresholds, padded rows (322) are; both equal the unfused props."""
    for w in (640, 322):
        clip = noise_clip(fmt, w, 90, seed=7)
        _dag_case(clip, lambda c: c.vszip.BoxBlur(hradius=1, vradius=1).vszip.PlaneMinMax(minthr=0.2, maxthr=0.3, clipb=c)
                  .vszip.PlaneAverage(exclude=[0], clipb=c))


@pytest.mark.parametrize("algorithm", [2, 1])
@pytest.mark.parametrize("fmt", ["YUV420P16", "GRAYS"])
def test_joint_bilateral_guided_by_a_blur_of_the_source(fmt, algorithm):
    clip = noise_clip(fmt, 322, 182, seed=8)
    args = dict(sigmaS=2, sigmaR=0.05, algorithm=algorithm)
    node, f = _dag_case(clip, lambda c: c.vszip.Bilateral(c, ref=c.vszip.BoxBlur(hradius=2, vradius=2), **args))
    assert [type(n.filter).__name__ for n in node._chain[0].nodes] == ["BoxBlurFilter", "BilateralFilter"]
    want = oa.bilateral(clip, ref=oa.boxblur(clip, hradius=2, vradius=2), **args)
    info = node.filter.info()
    _close(_planes(f), want["planes"], f"joint Bilateral {fmt} algorithm {algorithm}", exact=all(info.exact_lut[i] or not info.process[i] for i in range(3)))


def test_limitfilter_with_ref_from_inside_the_chain():
    clip = noise_clip("YUV420P16", 322, 182, seed=9)
    lf = dict(dark_thr=6, bright_thr=3, elast=2)

    def build(c):
        flt = c.vszip.BoxBlur(hradius=3, vradius=1)
        return flt.vszip.LimitFilter(c, ref=c.vszip.BoxBlur(hradius=1, vradius=3), **lf)
    node, f = _dag_case(clip, build)
    assert len(node._chain[0].nodes) == 3
    want = oa.limitfilter(oa.boxblur(clip, hradius=3, vradius=1), clip, oa.boxblur(clip, hradius=1, vradius=3), **lf)
    assert_same_planes(f.planes, want["planes"], "LimitFilter(flt, src, ref)")


def test_intermediate_read_three_elements_later():
    """a = BoxBlur(src) is read again by the LimitFilter three elements on, so the buffer plan keeps it alive past two pixel outputs."""
    clip = noise_clip("YUV420P16", 322, 182, seed=10)

    def build(c):
        a = c.vszip.BoxBlur(hradius=2, vradius=2)
        b = a.vszip.Limiter(min=[4096, 4096, 4096], max=[60000, 60000, 60000])
        d = b.vszip.BoxBlur(hradius=1, vradius=1).vszip.PlaneAverage(exclude=[0], clipb=a)
        return d.vszip.LimitFilter(a, dark_thr=8, bright_thr=8, elast=2)
    node, f = _dag_case(clip, build)
    a = oa.boxblur(clip, hradius=2, vradius=2)
    d = oa.boxblur(oa.limiter(a, min=[4096, 4096, 4096], max=[60000, 60000, 60000]), hradius=1, vradius=1)
    assert_same_planes(f.planes, oa.limitfilter(d, a, None, dark_thr=8, bright_thr=8, elast=2)["planes"], "read three elements later")
    _props_match(f.props, oa.planeaverage(d, [0], clipb=a))


def test_sixteen_elements_and_a_stats_only_dag():
    clip = noise_clip("GRAY16", 322, 182, seed=11)

    def build(c):
        x = c
        for k in range(7):
            x = x.vszip.BoxBlur(hradius=1 + k % 2, vradius=1).vszip.PlaneMinMax(clipb=c, prop=f"m{k}")
        return x.vszip.Limiter(min=[1000], max=[64000]).vszip.PlaneAverage(exclude=[0], clipb=c)
    node, f = _dag_case(clip, build)
    assert len(node._chain[0].nodes) == 16
    want = clip
    for k in range(7):
        want = oa.boxblur(want, hradius=1 + k % 2, vradius=1)
    want = oa.limiter(want, min=[1000], max=[64000])
    assert_same_planes(f.planes, want["planes"], "16 elements")
    # only statistics of the source against a blur of it: one frame up, nothing down
    node, f = _dag_case(clip, lambda c: c.vszip.PlaneMinMax(minthr=0.1, maxthr=0.1, clipb=c.vszip.BoxBlur(hradius=2, vradius=2)), down=False)
    _props_match(f.props, oa.planeminmax(clip, minthr=0.1, maxthr=0.1, clipb=oa.boxblur(clip, hradius=2, vradius=2)))


# --------------------------------------------------------------------------- PlaneMinMax + PlaneAverage with clipb from one read
@pytest.mark.parametrize("mm_args", [dict(minthr=0.1, maxthr=0.1), {}])
@pytest.mark.parametrize(("fmt", "w", "h", "n"), [("GRAY16", 3840, 2160, 2), ("GRAYS", 3840, 2160, 2), ("GRAYS", 3838, 2160, 3)])
def test_plane_stats_device_with_clipb(fmt, w, h, n, mm_args):
    a, b = vz.DeviceClip(fmt, w, h, n), vz.DeviceClip(fmt, w, h, n)
    a.fill_noise(seed=21)
    b.fill_noise(seed=22)
    mmf = vz.PlaneMinMaxFilter(a.info(), b.info(), **mm_args)
    avf = vz.PlaneAverageFilter(a.info(), b.info(), exclude=[0])
    sep_mm, sep_av = mmf.run_device(a, b), avf.run_device(a, b)
    got, fused = vz.plane_stats_device(mmf, avf, a, clipb=b)
    # float planes without row padding (3840 * 4 bytes) keep their two launches when thresholds are set (see DESIGN.md §4.4)
    assert fused == (fmt == "GRAY16" or not mm_args or w % 32 != 0), (fmt, w, mm_args)
    for i in range(n):
        want = dict(sep_mm[i])
        want.update(sep_av[i])
        assert got[i] == want, (i, got[i], want)
    if fused:
        assert all(g["psmDiff"] == s["psmDiff"] for g, s in zip(got, sep_mm))
    a.free()
    b.free()
