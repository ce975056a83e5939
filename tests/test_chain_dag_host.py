"""CPU-only: vszip_chain_create2 validates the graph it is given (filters are created without a device), and the Python mirror
turns clipb / ref / src inputs from inside a chain into the element lists it passes."""
import ctypes as C

import pytest

import vapoursynth_zip_b200 as vz

W, H = 64, 48


def _vi(fmt="GRAY16", w=W, h=H):
    return vz._vi(vz.FORMATS[fmt], w, h, 10)


def _create2(filters, inputs=None, second=None, third=None):
    n = len(filters)
    arr = lambda v: None if v is None else (C.c_int32 * n)(*v)
    h = vz.load_library().vszip_chain_create2((C.c_void_p * n)(*[f.handle for f in filters]), n, arr(inputs), arr(second), arr(third))
    if h:
        w = (C.c_int32 * 3)()
        vz.load_library().vszip_chain_planes(h, C.byref(w))
        vz.load_library().vszip_chain_free(h)
        return list(w)
    raise vz.Error(vz._last_error())


def test_create2_accepts_the_issue_graphs():
    vi = _vi()
    blur = vz.BoxBlurFilter(vi, hradius=2, vradius=2)
    mm = vz.PlaneMinMaxFilter(vi, vi, minthr=0.1, maxthr=0.1)
    av = vz.PlaneAverageFilter(vi, vi, exclude=[0])
    assert _create2([blur, mm, av], [0, 1, 1], [-1, 0, 0], [-1, -1, -1]) == [1, 0, 0]
    bil = vz.BilateralFilter(vi, vi, sigmaS=2, sigmaR=0.05)
    assert _create2([blur, bil], [0, 0], [-1, 1], None) == [1, 0, 0]
    lf = vz.LimitFilterFilter(vi, vi, vi, dark_thr=4)
    blur2 = vz.BoxBlurFilter(vi, hradius=1, vradius=3)
    assert _create2([blur, blur2, lf], [0, 0, 1], [-1, -1, 0], [-1, -1, 2]) == [1, 0, 0]
    # statistics of the source only: nothing differs from it
    assert _create2([blur, mm], [0, 0], [-1, 1]) == [0, 0, 0]


@pytest.mark.parametrize(("inputs", "second", "third", "msg"), [
    ([0, 2], [-1, 0], None, "chain: input[1] names filter 1, which does not come before filter 1"),
    ([0, 1], [-1, 2], None, "chain: second[1] names filter 1, which does not come before filter 1"),
    ([0, 3], [-1, 0], None, "chain: input[1] = 3 is out of range (0 = the source, k = the output of filter k - 1)"),
    ([0, 1], [-1, -2], None, "chain: second[1] = -2 is out of range (0 = the source, k = the output of filter k - 1)"),
    ([0, 1], [-1, -1], None, "chain: filter 1 (PlaneMinMax) was created with clipb; second[1] must name its input"),
    ([0, 1], [0, 0], None, "chain: filter 0 (BoxBlur) was created without a second clip; second[0] must be -1"),
    ([0, 1], [-1, 0], [-1, 0], "chain: filter 1 (PlaneMinMax) was created without a third clip; third[1] must be -1"),
])
def test_create2_rejects_bad_graphs(inputs, second, third, msg):
    vi = _vi()
    blur = vz.BoxBlurFilter(vi, hradius=2, vradius=2)
    mm = vz.PlaneMinMaxFilter(vi, vi)
    with pytest.raises(vz.Error) as e:
        _create2([blur, mm], inputs, second, third)
    assert str(e.value) == msg


def test_create2_rejects_stats_outputs_missing_inputs_and_formats():
    vi = _vi()
    mm = vz.PlaneMinMaxFilter(vi, None)
    blur = vz.BoxBlurFilter(vi)
    with pytest.raises(vz.Error, match=r"^chain: input\[1\] names filter 0 \(PlaneMinMax\), which has no pixel output$"):
        _create2([mm, blur], [0, 1])
    bil = vz.BilateralFilter(vi, vi, sigmaS=2)
    with pytest.raises(vz.Error, match=r"^chain: second\[1\] names filter 0 \(PlaneMinMax\), which has no pixel output$"):
        _create2([mm, bil], [0, 0], [-1, 1])
    lf = vz.LimitFilterFilter(vi, vi, None)
    with pytest.raises(vz.Error, match=r"^chain: filter 1 \(LimitFilter\) was created with src; second\[1\] must name its input$"):
        _create2([blur, lf], [0, 1], [-1, -1])
    with pytest.raises(vz.Error, match=r"^chain: filter 1 \(LimitFilter\) was created without ref; third\[1\] must be -1$"):
        _create2([blur, lf], [0, 1], [-1, 0], [-1, 0])
    other = vz.BoxBlurFilter(_vi("GRAY16", W + 2, H))
    with pytest.raises(vz.Error, match=r"^chain: filter 1 was created for a different video format than filter 0$"):
        _create2([blur, other], [0, 1])


def test_chain_create_still_rejects_second_clips():
    vi = _vi()
    lib = vz.load_library()
    fl = [vz.BoxBlurFilter(vi), vz.PlaneMinMaxFilter(vi, vi)]
    assert not lib.vszip_chain_create((C.c_void_p * 2)(*[f.handle for f in fl]), 2)
    assert vz._last_error() == "chain: filter 1 takes a second clip (ref/clipb); only single-input filters can be fused"


def test_python_builds_dag_chains():
    src = vz.core.BlankClip("GRAY16", W, H)
    # joint Bilateral guided by a blur of the source: the blur joins the chain as a side element
    blur = src.vszip.BoxBlur(hradius=2, vradius=2)
    bil = src.vszip.Bilateral(src, ref=blur, sigmaS=2, sigmaR=0.05)
    chain, source = vz._fusable_chain(bil)
    assert source is src and chain.nodes == [blur, bil] and chain.written == [True, False, False]
    # psmDiff pair against the source
    m = blur.vszip.PlaneMinMax(minthr=0.1, maxthr=0.1, clipb=src)
    a = m.vszip.PlaneAverage(exclude=[0], clipb=src)
    chain, source = vz._fusable_chain(a)
    assert source is src and chain.nodes == [blur, m, a]
    # a foreign clip ends the chain at its reader: the nodes after it still fuse, with it as their source
    other = vz.core.BlankClip("GRAY16", W, H)
    x = blur.vszip.PlaneMinMax(clipb=other)
    y = x.vszip.BoxBlur().vszip.Limiter(min=[0], max=[1000])
    chain, source = vz._fusable_chain(y)
    assert source is x and len(chain.nodes) == 2
    assert vz._fusable_chain(x) is None
