"""Fused chains that are small DAGs (vszip_chain_create2), end to end through the frame API with pinned host frames and T host
threads, against the same graphs evaluated as separate get_frame calls:
  4K GRAY16:      flt = src.BoxBlur(2, 2); m = flt.PlaneMinMax(0.1, 0.1, clipb=src); a = m.PlaneAverage([0], clipb=src)
  1080p YUV420P16: out = src.Bilateral(ref=src.BoxBlur(2, 2), sigmaS=2, sigmaR=0.05)
It prints frames/s and the frame bytes moved over PCIe per output frame (vszip_cuda_transfer_bytes), then the device-resident time
of PlaneMinMax + PlaneAverage with clipb on 4K GRAY16 and GRAYS frames: one read (vszip_planestats_device_b) against the two
separate reductions.
usage: python scripts/e2e_dag.py [frames] [threads]"""
import ctypes as C
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
import torch

import vapoursynth_zip_b200 as vz

NE = int(sys.argv[1]) if len(sys.argv) > 1 else 32
NT = int(sys.argv[2]) if len(sys.argv) > 2 else 8
vz.core.init([0])
lib = vz.load_library()
keep = []
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
print(f"GPU: {gpu or torch.cuda.get_device_name(0)}")


def pinned_frame(fmt, w, h, fill):
    f = vz.FORMATS[fmt]
    shapes = [f.plane_shape(w, h, p) for p in range(f.num_planes)]
    n = sum(a * b for a, b in shapes)
    t = torch.empty(n * np.dtype(f.dtype).itemsize, dtype=torch.uint8).pin_memory()
    a = t.numpy().view(f.dtype)
    if fill:
        a[:] = np.random.default_rng(len(keep)).integers(0, 1 << f.bits_per_sample, size=n, dtype=np.uint32).astype(f.dtype)
    keep.append(t)
    planes, off = [], 0
    for sh in shapes:
        planes.append(a[off:off + sh[0] * sh[1]].reshape(sh))
        off += sh[0] * sh[1]
    return planes


def run(fn, reps=3):
    with ThreadPoolExecutor(NT) as ex:
        list(ex.map(fn, range(NE)))
        b0 = vz.core.transfer_bytes()
        t0 = time.perf_counter()
        for _ in range(reps):
            list(ex.map(fn, range(NE)))
        dt = time.perf_counter() - t0
        b1 = vz.core.transfer_bytes()
    return reps * NE / dt, (b1[0] - b0[0] + b1[1] - b0[1]) / (reps * NE) / 1e6


def chain(filters, inputs, second):
    n = len(filters)
    h = lib.vszip_chain_create2((C.c_void_p * n)(*[f.handle for f in filters]), n, (C.c_int32 * n)(*inputs), (C.c_int32 * n)(*second), None)
    assert h, vz._last_error()
    return h


def ok(rc):
    assert rc == 0, vz._last_error()


def case_stats():
    fmt, w, h = "GRAY16", 3840, 2160
    vi = vz._vi(vz.FORMATS[fmt], w, h, 5000)
    blur = vz.BoxBlurFilter(vi, hradius=2, vradius=2)
    mm = vz.PlaneMinMaxFilter(vi, vi, minthr=0.1, maxthr=0.1)
    av = vz.PlaneAverageFilter(vi, vi, exclude=[0])
    src = [vz._cframe(pinned_frame(fmt, w, h, True)) for _ in range(NE)]
    mid = [vz._cframe(pinned_frame(fmt, w, h, False)) for _ in range(NE)]
    dst = [vz._cframe(pinned_frame(fmt, w, h, False)) for _ in range(NE)]
    props = {}

    def unfused(i):
        pm, pa = vz._MinMaxProps(), vz._AverageProps()
        ok(lib.vszip_boxblur_get_frame(blur.handle, i, C.byref(src[i]), C.byref(mid[i])))
        ok(lib.vszip_planeminmax_get_frame(mm.handle, i, C.byref(mid[i]), C.byref(src[i]), C.byref(pm)))
        ok(lib.vszip_planeaverage_get_frame(av.handle, i, C.byref(mid[i]), C.byref(src[i]), C.byref(pa)))
        props[("u", i)] = (vz.PlaneMinMaxFilter.to_props(pm), vz.PlaneAverageFilter.to_props(pa))

    ch = chain([blur, mm, av], [0, 1, 1], [-1, 0, 0])

    def fused(i):
        pm, pa = vz._MinMaxProps(), vz._AverageProps()
        ok(lib.vszip_chain_get_frame(ch, i, C.byref(src[i]), C.byref(dst[i]),
                                     (C.c_void_p * 3)(None, C.cast(C.pointer(pm), C.c_void_p), C.cast(C.pointer(pa), C.c_void_p))))
        props[("f", i)] = (vz.PlaneMinMaxFilter.to_props(pm), vz.PlaneAverageFilter.to_props(pa))

    fa, ma = run(unfused)
    fb, mb = run(fused)
    same = all(props[("u", i)] == props[("f", i)] for i in range(NE)) and all(
        np.array_equal(np.ctypeslib.as_array(C.cast(mid[i].data[0], C.POINTER(C.c_uint16)), (h, w)),
                       np.ctypeslib.as_array(C.cast(dst[i].data[0], C.POINTER(C.c_uint16)), (h, w))) for i in range(2))
    print(f"BoxBlur(2,2) -> PlaneMinMax(0.1,0.1,clipb=src) -> PlaneAverage([0],clipb=src), {w}x{h} {fmt}, {NT} host threads, pinned: "
          f"separate {fa:.0f} fps ({ma:.1f} MB/frame over PCIe), fused chain {fb:.0f} fps ({mb:.1f} MB/frame), {fb / fa:.2f}x, same results: {same}")
    lib.vszip_chain_free(ch)


def case_bilateral():
    fmt, w, h = "YUV420P16", 1920, 1080
    vi = vz._vi(vz.FORMATS[fmt], w, h, 5000)
    blur = vz.BoxBlurFilter(vi, hradius=2, vradius=2)
    bil = vz.BilateralFilter(vi, vi, sigmaS=2, sigmaR=0.05)
    src = [pinned_frame(fmt, w, h, True) for _ in range(NE)]
    mid = [pinned_frame(fmt, w, h, False) for _ in range(NE)]
    dst = [pinned_frame(fmt, w, h, False) for _ in range(NE)]
    fs, fm, fd = ([vz._cframe(p) for p in fr] for fr in (src, mid, dst))

    def unfused(i):
        ok(lib.vszip_boxblur_get_frame(blur.handle, i, C.byref(fs[i]), C.byref(fm[i])))
        ok(lib.vszip_bilateral_get_frame(bil.handle, i, C.byref(fs[i]), C.byref(fm[i]), C.byref(fd[i])))

    ch = chain([blur, bil], [0, 0], [-1, 1])

    def fused(i):
        ok(lib.vszip_chain_get_frame(ch, i, C.byref(fs[i]), C.byref(fd[i]), (C.c_void_p * 2)(None, None)))

    fa, ma = run(unfused)
    ref_out = [[p.copy() for p in d] for d in dst[:2]]
    for d in dst:
        for p in d:
            p[:] = 0
    fb, mb = run(fused)
    same = all(np.array_equal(a, b) for i in range(2) for a, b in zip(dst[i], ref_out[i]))
    print(f"Bilateral(src, ref=BoxBlur(src,2,2), sigmaS=2, sigmaR=0.05), {w}x{h} {fmt}, {NT} host threads, pinned: separate {fa:.0f} fps "
          f"({ma:.1f} MB/frame over PCIe), fused chain {fb:.0f} fps ({mb:.1f} MB/frame), {fb / fa:.2f}x, outputs identical: {same}")
    lib.vszip_chain_free(ch)


def device_stats(fmt, mm_args, n=64, reps=20):
    w, h = 3840, 2160
    a, b = vz.DeviceClip(fmt, w, h, n), vz.DeviceClip(fmt, w, h, n)
    a.fill_noise(seed=1)
    b.fill_noise(seed=2)
    mm = vz.PlaneMinMaxFilter(a.info(), b.info(), **mm_args)
    av = vz.PlaneAverageFilter(a.info(), b.info(), exclude=[0])
    fused = C.c_int32(0)

    def one():
        ok(lib.vszip_planestats_device_b(mm.handle, av.handle, a.handle, b.handle, 0, n, None, None, C.byref(fused), None))

    def two():
        ok(lib.vszip_planeminmax_device(mm.handle, a.handle, b.handle, 0, n, None, None))
        ok(lib.vszip_planeaverage_device(av.handle, a.handle, b.handle, 0, n, None, None))

    out = {}
    for name, fn in (("one read", one), ("two launches", two)) * 2:  # alternated, the second round is reported
        fn()
        vz.core.sync()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        vz.core.sync()
        out[name] = (time.perf_counter() - t0) / (reps * n) * 1e6
    gbs = 2 * w * h * vz.FORMATS[fmt].bytes_per_sample / (out["one read"] * 1e-6) / 1e9
    print(f"PlaneMinMax{mm_args or '(no thresholds)'} + PlaneAverage([0]) with clipb, {w}x{h} {fmt}, {n} device-resident frames: "
          f"one read {out['one read']:.1f} us/frame ({gbs:.0f} GB/s of a+b), two launches {out['two launches']:.1f} us/frame "
          f"({out['two launches'] / out['one read']:.2f}x); fused route: {bool(fused.value)}")
    a.free()
    b.free()


case_stats()
case_bilateral()
device_stats("GRAY16", dict(minthr=0.1, maxthr=0.1))
device_stats("GRAY16", {})
device_stats("GRAYS", {})
device_stats("GRAYS", dict(minthr=0.1, maxthr=0.1))
