"""CPU-only: what every vszip node hands the library and what it makes of the answer.  `vz._lib` is swapped for a proxy that
forwards to the real library but records vszip_cuda_init, every `vszip_*_get_frame` and vszip_chain_get_frame instead of running
them, and fills stats props structs with fixed values.  For each namespace function, bound and unbound, this pins which clip's
processed planes reach which argument and for which frame, fresh versus shared output planes and the resulting props; for the
fused graph shapes of test_gpu_chain.py and test_gpu_chain_dag.py it pins the vszip_chain_create2 arrays and the fused props.

Frame arguments are recorded as plane labels: "a2.1" is plane 1 of frame 2 of source clip a, "dst" a plane the library would
write, None a NULL pointer.  Input frames are recorded on the planes the filter processes only: the library reads no others."""
import ctypes as C

import numpy as np
import pytest

import vapoursynth_zip_b200 as vz

W, H = 64, 32
STATS = {"planeminmax": vz._MinMaxProps, "planeaverage": vz._AverageProps}


class Recorder:
    """Stands in for vz._lib: forwards every symbol to the real library except the ones that would need a GPU."""

    def __init__(self, real):
        self.real, self.labels = real, {}
        self.calls, self.inits, self.filled, self.kinds, self.chains, self.dst = [], 0, 0, {}, {}, set()

    def __getattr__(self, name):
        real = getattr(self.real, name)
        if name == "vszip_cuda_init":
            return self._init
        if name == "vszip_chain_create2":
            return lambda fl, n, *arrs: self._chain_create(real, fl, n, arrs)
        if name.endswith("_create") and name != "vszip_chain_create":
            return lambda *a: self._created(name[len("vszip_"):-len("_create")], real(*a))
        if name == "vszip_chain_get_frame":
            return self._chain_get_frame
        if name.endswith("_get_frame"):
            return lambda h, n, *args: self._get_frame(name[len("vszip_"):-len("_get_frame")], h, n, args)
        return real

    def _init(self, devices, count):
        self.inits += 1
        return 1

    def _created(self, kind, h):
        if h:
            self.kinds[h] = kind
        return h

    def _chain_create(self, real, fl, n, arrs):
        h = real(fl, n, *arrs)
        if h:
            handles = [fl[i] for i in range(n)]
            inputs, second, third = ([-2] * n if a is None else list(a) for a in arrs)
            self.chains[h] = (handles, second)
            self.calls.append(("create2", [self.kinds[x] for x in handles], inputs, second, third))
        return h

    def _process(self, h):
        mask = (C.c_int32 * 3)()
        self.real.vszip_filter_planes(h, C.byref(mask))
        return [bool(m) for m in mask]

    def _frame(self, ref, mask=(True, True, True), dst=False):
        if ref is None:
            return None
        fr = ref._obj
        out = []
        for i in range(3):
            d = fr.data[i]
            if not d or not mask[i]:
                out.append(None)
            elif d in self.labels:
                out.append(self.labels[d])
            elif dst or d in self.dst:
                self.dst.add(d)
                out.append("dst")
            else:
                out.append("?")
        return out

    def _fill(self, props, kind, process, has_diff):
        self.filled += 1
        k = self.filled
        props.count = sum(process)
        props.has_diff = int(has_diff)
        for i in range(props.count):
            props.plane[i] = [p for p in range(3) if process[p]][i]
            props.diff[i] = k + i / 4
            if kind == "planeminmax":
                props.is_float = 0
                props.imin[i], props.imax[i] = 10 * k + i, 10 * k + 5 + i
            else:
                props.avg[i] = k + 0.5 + i / 4

    def _get_frame(self, kind, h, n, args):
        *frames, out = args
        process = self._process(h)
        if kind in STATS:
            self._fill(out._obj, kind, process, frames[1] is not None)
            rec = "props"
        else:
            rec = self._frame(out, dst=True)
        self.calls.append((kind, n, [self._frame(f, process) for f in frames], rec))
        return 0

    def _chain_get_frame(self, h, n, src, dst, props_out):
        handles, second = self.chains[h]
        for i, x in enumerate(handles):
            if self.kinds[x] in STATS:
                struct = STATS[self.kinds[x]]
                self._fill(C.cast(props_out[i], C.POINTER(struct)).contents, self.kinds[x], self._process(x), second[i] >= 0)
        self.calls.append(("chain", n, self._frame(src), self._frame(dst, dst=True)))
        return 0

    def source(self, tag, fmt, frames=4, props=None):
        """A clip whose every plane of every frame is its own array, so a pointer names clip, frame and plane."""
        f = vz.FORMATS[fmt]
        planes = [[np.full(f.plane_shape(W, H, p), 3 * n + p, f.dtype) for p in range(f.num_planes)] for n in range(frames)]
        for n, fr in enumerate(planes):
            for p, a in enumerate(fr):
                self.labels[a.ctypes.data] = f"{tag}{n}.{p}"
        return vz.core.clip_from_frames(fmt, planes, dict(props or {}, tag=tag))

    def planes(self, frame):
        """Output planes: a source plane they share, or "dst" for one the library wrote."""
        return [self.labels.get(p.ctypes.data) or ("dst" if p.ctypes.data in self.dst else "?") for p in frame.planes]


@pytest.fixture
def rec():
    real = vz.load_library()
    r = Recorder(real)
    saved = vz._lib, vz.core._ready, vz.core.fuse_chains
    vz._lib, vz.core._ready, vz.core.fuse_chains = r, False, True
    try:
        yield r
    finally:
        vz._lib, vz.core._ready, vz.core.fuse_chains = saved


# --------------------------------------------------------------------------- one node on source clips
def _sources(rec):
    a = rec.source("a", "YUV420P16", props={"_ColorRange": 0, "psmDiff": -1.0, "xMin": -2, "psmAvg": 7.0})
    b = rec.source("b", "YUV420P16", frames=6)
    c = rec.source("c", "YUV420P16")
    d = rec.source("d", "YUV420P16", props={"_ColorRange": 1})
    g = rec.source("g", "YUV420P8", props={"_ColorRange": 1, "psmMin": 3})
    h = rec.source("h", "YUV420P8", frames=6, props={"_ColorRange": 1, "hue": 1})
    return dict(a=a, b=b, c=c, d=d, g=g, h=h, core=vz.core)


NODES = {
    "BoxBlur": [lambda a, **_: a.vszip.BoxBlur(planes=[1, 2], hradius=1, vradius=1),
                lambda a, core, **_: core.vszip.BoxBlur(a, [1, 2], 1, None, 1)],
    "Limiter": [lambda a, **_: a.vszip.Limiter(planes=[0]),
                lambda a, core, **_: core.vszip.Limiter(clip=a, planes=[0])],
    "Bilateral": [lambda a, b, **_: a.vszip.Bilateral(ref=b, sigmaS=2, planes=[0]),
                  lambda a, b, core, **_: core.vszip.Bilateral(a, b, 2, planes=[0])],
    "Bilateral/no ref": [lambda a, **_: a.vszip.Bilateral(sigmaS=2, planes=[0, 2]),
                         lambda a, core, **_: core.vszip.Bilateral(a, sigmaS=2, planes=[0, 2])],
    "PlaneMinMax": [lambda a, b, **_: a.vszip.PlaneMinMax(clipb=b, planes=[0, 2], prop="x"),
                    lambda a, b, core, **_: core.vszip.PlaneMinMax(a, None, None, b, [0, 2], "x")],
    "PlaneMinMax/no clipb": [lambda a, **_: a.vszip.PlaneMinMax(),
                             lambda a, core, **_: core.vszip.PlaneMinMax(clipa=a)],
    "PlaneAverage": [lambda a, b, **_: a.vszip.PlaneAverage(exclude=[0], clipb=b),
                     lambda a, b, core, **_: core.vszip.PlaneAverage(a, [0], b)],
    "PlaneAverage/no clipb": [lambda a, **_: a.vszip.PlaneAverage(exclude=[0], planes=[1, 2], prop="y"),
                              lambda a, core, **_: core.vszip.PlaneAverage(clipa=a, exclude=[0], planes=[1, 2], prop="y")],
    "LimitFilter": [lambda a, c, d, **_: a.vszip.LimitFilter(c, d, dark_thr=4, planes=[0, 1]),
                    lambda a, c, d, core, **_: core.vszip.LimitFilter(a, c, d, 4, planes=[0, 1])],
    "LimitFilter/no ref": [lambda c, d, **_: d.vszip.LimitFilter(c, dark_thr=4),
                           lambda c, d, core, **_: core.vszip.LimitFilter(src=c, flt=d, dark_thr=4)],
    "AdaptiveBinarize": [lambda g, h, **_: g.vszip.AdaptiveBinarize(h, c=2),
                         lambda g, h, core, **_: core.vszip.AdaptiveBinarize(clip2=h, clip=g)],
}


# (calls, output planes, props[, LimitFilter's dark_thr after the _ColorRange of flt's frame 0])
NODE_RESULTS = {
    "BoxBlur": (
        [("boxblur", 2, [[None, "a2.1", "a2.2"]], [None, "dst", "dst"])],
        ["a2.0", "dst", "dst"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a")],
    ),
    "Limiter": (
        [("limiter", 2, [["a2.0", None, None]], ["dst", None, None])],
        ["dst", "a2.1", "a2.2"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a")],
    ),
    "Bilateral": (
        [("bilateral", 2, [["a2.0", None, None], ["b2.0", None, None]], ["dst", None, None])],
        ["dst", "a2.1", "a2.2"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a")],
    ),
    "Bilateral/no ref": (
        [("bilateral", 2, [["a2.0", None, "a2.2"], None], ["dst", None, "dst"])],
        ["dst", "a2.1", "dst"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a")],
    ),
    "PlaneMinMax": (
        [("planeminmax", 2, [["a2.0", None, "a2.2"], ["b2.0", None, "b2.2"]], "props")],
        ["a2.0", "a2.1", "a2.2"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("psmAvg", 7.0), ("tag", "a"), ("xMin", [10, 11]), ("xMax", [15, 16]), ("xDiff", [1.0, 1.25])],
    ),
    "PlaneMinMax/no clipb": (
        [("planeminmax", 2, [["a2.0", None, None], None], "props")],
        ["a2.0", "a2.1", "a2.2"],
        [("_ColorRange", 0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a"), ("psmMin", 10), ("psmMax", 15)],
    ),
    "PlaneAverage": (
        [("planeaverage", 2, [["a2.0", None, None], ["b2.0", None, None]], "props")],
        ["a2.0", "a2.1", "a2.2"],
        [("_ColorRange", 0), ("xMin", -2), ("tag", "a"), ("psmAvg", 1.5), ("psmDiff", 1.0)],
    ),
    "PlaneAverage/no clipb": (
        [("planeaverage", 2, [[None, "a2.1", "a2.2"], None], "props")],
        ["a2.0", "a2.1", "a2.2"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a"), ("yAvg", [1.5, 1.75])],
    ),
    "LimitFilter": (
        [("limitfilter", 2, [["a2.0", "a2.1", None], ["c2.0", "c2.1", None], ["d2.0", "d2.1", None]], ["dst", "dst", None])],
        ["dst", "dst", "a2.2"],
        [("_ColorRange", 0), ("psmDiff", -1.0), ("xMin", -2), ("psmAvg", 7.0), ("tag", "a")],
        [1028.0, 1028.0, 1028.0],
    ),
    "LimitFilter/no ref": (
        [("limitfilter", 2, [["d2.0", "d2.1", "d2.2"], ["c2.0", "c2.1", "c2.2"], None], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("tag", "d")],
        [1024.0, 1024.0, 1024.0],
    ),
    "AdaptiveBinarize": (
        [("adaptivebinarize", 2, [["g2.0", "g2.1", "g2.2"], ["h2.0", "h2.1", "h2.2"]], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 0), ("psmMin", 3), ("tag", "g")],
    ),
}


@pytest.mark.parametrize("name", list(NODES))
def test_single_node(rec, name):
    src = _sources(rec)
    got = []
    for build in NODES[name]:
        rec.calls, rec.filled = [], 0
        node = build(**src)
        frame = node.get_frame(2)
        got.append((rec.calls, rec.planes(frame), list(frame.props.items())))
        if name.startswith("LimitFilter"):
            got[-1] += (node.filter.info()["dark_thr"],)
    assert got[0] == NODE_RESULTS[name]
    assert got[1] == got[0]
    assert rec.inits == 1


# --------------------------------------------------------------------------- fused chains
def _s(rec, fmt):
    return rec.source("s", fmt, props={"_ColorRange": 1, "psmMin": -5})


def _limitfilter_ref(c):
    ref = c.vszip.BoxBlur(hradius=1, vradius=3)
    return c.vszip.BoxBlur(hradius=3, vradius=1).vszip.LimitFilter(c, ref=ref, dark_thr=6, bright_thr=3, elast=2)


def _intermediate(c):
    a = c.vszip.BoxBlur(hradius=2, vradius=2)
    b = a.vszip.Limiter(min=[4096, 4096, 4096], max=[60000, 60000, 60000])
    d = b.vszip.BoxBlur(hradius=1, vradius=1).vszip.PlaneAverage(exclude=[0], clipb=a)
    return d.vszip.LimitFilter(a, dark_thr=8, bright_thr=8, elast=2)


def _sixteen(c):
    x = c
    for k in range(7):
        x = x.vszip.BoxBlur(hradius=1 + k % 2, vradius=1).vszip.PlaneMinMax(clipb=c, prop=f"m{k}")
    return x.vszip.Limiter(min=[1000], max=[64000]).vszip.PlaneAverage(exclude=[0], clipb=c)


def _cut(c, other):
    x = c.vszip.BoxBlur(hradius=2, vradius=2).vszip.PlaneMinMax(clipb=other)
    return x.vszip.BoxBlur().vszip.Limiter(min=[0], max=[1000])


SHAPES = {
    "config5": ("YUV444PS", lambda c, o: c.vszip.BoxBlur(hradius=13, vradius=13).vszip.Bilateral(sigmaS=2, sigmaR=2)
                .vszip.PlaneMinMax(minthr=0.1, maxthr=0.1, planes=[0])),
    "partial planes": ("YUV420P16", lambda c, o: c.vszip.BoxBlur(planes=[0], hradius=3, hpasses=2, vradius=0, vpasses=0)
                       .vszip.PlaneAverage(exclude=[0, 7], planes=[0, 1, 2], prop="a")
                       .vszip.Bilateral(sigmaS=1.5, sigmaR=0.02, planes=[1, 2])
                       .vszip.PlaneMinMax(minthr=0.05, maxthr=0.2, planes=[0, 2], prop="b")
                       .vszip.BoxBlur(planes=[2], hradius=0, hpasses=0, vradius=5, vpasses=3)),
    "stats only": ("GRAY16", lambda c, o: c.vszip.PlaneMinMax(minthr=0.1).vszip.PlaneAverage(exclude=[5])),
    "pbfic": ("GRAY16", lambda c, o: c.vszip.Bilateral(sigmaS=3, sigmaR=0.1, algorithm=1).vszip.BoxBlur(hradius=2, vradius=2)),
    "foreign clipb": ("GRAY8", lambda c, o: c.vszip.BoxBlur().vszip.PlaneMinMax(clipb=o)),
    "diamond": ("YUV420P16", lambda c, o: c.vszip.BoxBlur(hradius=2, vradius=2)
                .vszip.LimitFilter(c, dark_thr=[16, 4], bright_thr=[8, 4], elast=[3, 2], planes=[0, 2])
                .vszip.PlaneMinMax(minthr=0.05, maxthr=0.05)),
    "diamond after three": ("GRAYS", lambda c, o: c.vszip.BoxBlur(hradius=1, vradius=1).vszip.BoxBlur(hradius=3, vradius=0, vpasses=0)
                            .vszip.Limiter(min=[0.1], max=[0.9]).vszip.LimitFilter(c, dark_thr=8, bright_thr=8, elast=1.5)),
    "adaptive binarize": ("YUV420P8", lambda c, o: c.vszip.AdaptiveBinarize(c.vszip.BoxBlur(hradius=5, vradius=5), c=2)),
    "foreign src": ("GRAY16", lambda c, o: c.vszip.BoxBlur(hradius=2, vradius=2).vszip.LimitFilter(o, dark_thr=8)),
    "foreign ref": ("GRAY16", lambda c, o: c.vszip.BoxBlur(hradius=2, vradius=2).vszip.LimitFilter(c, o, dark_thr=8)),
    "props follow clip": ("GRAY8", lambda c, o: c.vszip.AdaptiveBinarize(c.vszip.BoxBlur(hradius=3, vradius=3).vszip.PlaneMinMax(minthr=0.1),
                                                                         c=1)),
    "minmax against the source": ("GRAY16", lambda c, o: c.vszip.BoxBlur(hradius=2, vradius=2)
                                  .vszip.PlaneMinMax(clipb=c, minthr=0.1, maxthr=0.1)),
    "clipb pair": ("YUV420P16", lambda c, o: c.vszip.BoxBlur(hradius=2, vradius=2)
                   .vszip.PlaneMinMax(minthr=0.1, maxthr=0.1, clipb=c, planes=[0, 1, 2])
                   .vszip.PlaneAverage(exclude=[0], clipb=c, planes=[0, 1, 2], prop="a")),
    "joint bilateral": ("YUV420P16", lambda c, o: c.vszip.Bilateral(c, ref=c.vszip.BoxBlur(hradius=2, vradius=2), sigmaS=2, sigmaR=0.05)),
    "limitfilter ref": ("YUV420P16", lambda c, o: _limitfilter_ref(c)),
    "intermediate": ("YUV420P16", lambda c, o: _intermediate(c)),
    "sixteen": ("GRAY16", lambda c, o: _sixteen(c)),
    "stats-only dag": ("GRAY16", lambda c, o: c.vszip.PlaneMinMax(minthr=0.1, maxthr=0.1, clipb=c.vszip.BoxBlur(hradius=2, vradius=2))),
    "cut": ("GRAY16", _cut),
}


# (calls, output planes, props) of frame 1; the unfused calls at frame 0 are LimitFilter reading the _ColorRange of flt
SHAPE_RESULTS = {
    "config5": (
        [("create2", ["boxblur", "bilateral", "planeminmax"], [0, 1, 2], [-1, -1, -1], [-1, -1, -1]),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15)],
    ),
    "partial planes": (
        [("create2", ["boxblur", "planeaverage", "bilateral", "planeminmax", "boxblur"], [0, 1, 1, 3, 3], [-1] * 5, [-1] * 5),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s"), ("aAvg", [1.5, 1.75, 2.0]), ("bMin", [20, 21]), ("bMax", [25, 26])],
    ),
    "stats only": (
        [("create2", ["planeminmax", "planeaverage"], [0, 0], [-1, -1], [-1, -1]),
         ("chain", 1, ["s1.0", None, None], [None, None, None])],
        ["s1.0"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15), ("psmAvg", 2.5)],
    ),
    "pbfic": (
        [("create2", ["bilateral", "boxblur"], [0, 1], [-1, -1], [-1, -1]),
         ("chain", 1, ["s1.0", None, None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")],
    ),
    "foreign clipb": (
        [("boxblur", 1, [["s1.0", None, None]], ["dst", None, None]),
         ("planeminmax", 1, [["dst", None, None], ["o1.0", None, None]], "props")],
        ["dst"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15), ("psmDiff", 1.0)],
    ),
    "diamond": (
        [("boxblur", 0, [["s0.0", "s0.1", "s0.2"]], ["dst", "dst", "dst"]),
         ("create2", ["boxblur", "limitfilter", "planeminmax"], [0, 1, 2], [-1, 0, -1], [-1, -1, -1]),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15)],
    ),
    "diamond after three": (
        [("create2", ["boxblur", "boxblur", "limiter"], [0, 1, 2], [-1, -1, -1], [-1, -1, -1]),
         ("chain", 0, ["s0.0", None, None], ["dst", None, None]),
         ("create2", ["boxblur", "boxblur", "limiter", "limitfilter"], [0, 1, 2, 3], [-1, -1, -1, 0], [-1, -1, -1, -1]),
         ("chain", 1, ["s1.0", None, None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")],
    ),
    "adaptive binarize": (
        [("create2", ["boxblur", "adaptivebinarize"], [0, 1], [-1, 0], [-1, -1]),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 0), ("psmMin", -5), ("tag", "s")],
    ),
    "foreign src": (
        [("boxblur", 0, [["s0.0", None, None]], ["dst", None, None]),
         ("boxblur", 1, [["s1.0", None, None]], ["dst", None, None]),
         ("limitfilter", 1, [["dst", None, None], ["o1.0", None, None], None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")],
    ),
    "foreign ref": (
        [("boxblur", 0, [["s0.0", None, None]], ["dst", None, None]),
         ("boxblur", 1, [["s1.0", None, None]], ["dst", None, None]),
         ("limitfilter", 1, [["dst", None, None], ["s1.0", None, None], ["o1.0", None, None]], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")],
    ),
    "props follow clip": (
        [("create2", ["boxblur", "planeminmax", "adaptivebinarize"], [0, 1, 1], [-1, -1, 0], [-1, -1, -1]),
         ("chain", 1, ["s1.0", None, None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 0), ("psmMin", -5), ("tag", "s")],
    ),
    "minmax against the source": (
        [("create2", ["boxblur", "planeminmax"], [0, 1], [-1, 0], [-1, -1]),
         ("chain", 1, ["s1.0", None, None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15), ("psmDiff", 1.0)],
    ),
    "clipb pair": (
        [("create2", ["boxblur", "planeminmax", "planeaverage"], [0, 1, 1], [-1, 0, 0], [-1, -1, -1]),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", [10, 11, 12]), ("psmMax", [15, 16, 17]), ("psmDiff", [1.0, 1.25, 1.5]),
         ("aAvg", [2.5, 2.75, 3.0]), ("aDiff", [2.0, 2.25, 2.5])],
    ),
    "joint bilateral": (
        [("create2", ["boxblur", "bilateral"], [0, 0], [-1, 1], [-1, -1]),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")],
    ),
    "limitfilter ref": (
        [("boxblur", 0, [["s0.0", "s0.1", "s0.2"]], ["dst", "dst", "dst"]),
         ("create2", ["boxblur", "boxblur", "limitfilter"], [0, 0, 1], [-1, -1, 0], [-1, -1, 2]),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")],
    ),
    "intermediate": (
        [("create2", ["boxblur", "limiter", "boxblur", "planeaverage"], [0, 1, 2, 3], [-1, -1, -1, 1], [-1, -1, -1, -1]),
         ("chain", 0, ["s0.0", "s0.1", "s0.2"], ["dst", "dst", "dst"]),
         ("create2", ["boxblur", "limiter", "boxblur", "planeaverage", "limitfilter"], [0, 1, 2, 3, 3], [-1, -1, -1, 1, 1], [-1] * 5),
         ("chain", 1, ["s1.0", "s1.1", "s1.2"], ["dst", "dst", "dst"])],
        ["dst", "dst", "dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s"), ("psmAvg", 2.5), ("psmDiff", 2.0)],
    ),
    "sixteen": (
        [("create2", ["boxblur", "planeminmax"] * 7 + ["limiter", "planeaverage"], [0] + [k for k in range(1, 15, 2) for _ in "ab"] + [15],
          [-1, 0] * 8, [-1] * 16),
         ("chain", 1, ["s1.0", None, None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("psmMin", -5), ("tag", "s")]
        + [(f"m{k}{key}", v) for k in range(7) for key, v in (("Min", 10 * k + 10), ("Max", 10 * k + 15), ("Diff", k + 1.0))]
        + [("psmAvg", 8.5), ("psmDiff", 8.0)],
    ),
    "stats-only dag": (
        [("create2", ["boxblur", "planeminmax"], [0, 0], [-1, 1], [-1, -1]),
         ("chain", 1, ["s1.0", None, None], [None, None, None])],
        ["s1.0"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15), ("psmDiff", 1.0)],
    ),
    "cut": (
        [("create2", ["boxblur", "limiter"], [0, 1], [-1, -1], [-1, -1]),
         ("boxblur", 1, [["s1.0", None, None]], ["dst", None, None]),
         ("planeminmax", 1, [["dst", None, None], ["o1.0", None, None]], "props"),
         ("chain", 1, ["dst", None, None], ["dst", None, None])],
        ["dst"],
        [("_ColorRange", 1), ("tag", "s"), ("psmMin", 10), ("psmMax", 15), ("psmDiff", 1.0)],
    ),
}


@pytest.mark.parametrize("name", list(SHAPES))
def test_fused_shape(rec, name):
    fmt, build = SHAPES[name]
    c, o = _s(rec, fmt), rec.source("o", fmt)
    node = build(c, o)
    frame = node.get_frame(1)
    assert (rec.calls, rec.planes(frame), list(frame.props.items())) == SHAPE_RESULTS[name]


def test_limitfilter_checks_arguments_before_reading_frame_0(rec):
    """LimitFilter creates its filter, reads the _ColorRange of flt's frame 0 and creates it again: a bad argument is reported
    before any frame of flt is computed."""
    src = _sources(rec)
    flt = src["a"].vszip.BoxBlur(hradius=1, vradius=1)
    with pytest.raises(vz.Error, match="^LimitFilter: dark_thr value -1 is below minimum 0"):
        flt.vszip.LimitFilter(src["c"], dark_thr=-1)
    with pytest.raises(vz.Error, match="^LimitFilter: flt and src are required$"):
        flt.vszip.LimitFilter(ref=src["c"])
    with pytest.raises(vz.Error, match="^AdaptiveBinarize: clip and clip2 are required$"):
        vz.core.vszip.AdaptiveBinarize(src["g"])
    assert rec.calls == []
    flt.vszip.LimitFilter(src["c"], dark_thr=4)
    assert rec.calls == [("boxblur", 0, [["a0.0", "a0.1", "a0.2"]], ["dst", "dst", "dst"])]
