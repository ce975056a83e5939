"""Secondary measurements: the other BASELINE.json configs, device-resident, CUDA-event timed.
Not the contract line (bench.py prints that); results go to stdout as JSON and, with --out, to a file.
usage: python scripts/bench_extras.py [--frames N] [--reps R] [--only REGEX] [--out profiles/bench_extras_rXX.json]
--only clahe: the CLAHE group (device batches, get_frame on pinned frames, and OpenCV on every host core for comparison);
--only colormap: the same for ColorMap; --only packrgb: the same for PackRGB, next to a numpy pack on every host core."""
import argparse
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import numpy as np
import torch

import vapoursynth_zip_b200 as vz

ap = argparse.ArgumentParser()
ap.add_argument("--frames", type=int, default=128)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--out", default=None)
ap.add_argument("--only", default=None, help="regex: run only the configurations whose name matches")
args = ap.parse_args()

vz.core.init([0])
st = torch.cuda.Stream()
torch.cuda.set_stream(st)
PEAK = json.loads((Path(__file__).resolve().parents[1] / "MEASURED_PEAKS.json").read_text())["hbm_gbs"] if (Path(__file__).resolve().parents[1] / "MEASURED_PEAKS.json").exists() else 6650.0


def timed(fn, reps):
    for _ in range(2):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


results = []


def record(name, fmt, w, h, frames, algo_bytes_per_frame, ms):
    fps = frames / (ms * 1e-3)
    gbs = algo_bytes_per_frame * fps / 1e9
    results.append({"config": name, "format": fmt, "size": f"{w}x{h}", "frames_per_launch": frames, "ms_per_launch": ms, "fps": fps,
                    "us_per_frame": ms * 1e3 / frames, "algorithmic_bytes_per_frame": algo_bytes_per_frame, "algorithmic_GBps": gbs,
                    "frac_of_measured_hbm_peak": gbs / PEAK})
    print(f"{name:58s} {fps:12.0f} fps  {ms * 1e3 / frames:8.2f} us/frame  {gbs:8.1f} GB/s  {100 * gbs / PEAK:5.1f}% of {PEAK:.0f}", file=sys.stderr)


def skip(name):
    import re
    return args.only is not None and not re.search(args.only, name)


def pixel_cfg(name, fmt, w, h, frames, make_filter, noise=True):
    if skip(name):
        return
    src, dst = vz.DeviceClip(fmt, w, h, frames), vz.DeviceClip(fmt, w, h, frames)
    if noise:
        src.fill_noise(1234)
    f = make_filter(src)
    ms = timed(lambda: f.run_device(src, dst, first=0, count=frames, stream=st.cuda_stream), args.reps)
    record(name, fmt, w, h, frames, 2 * src.frame_bytes, ms)
    src.free(); dst.free()


def multi_cfg(name, fmt, w, h, frames, nin, run, prep=None):
    """pointwise filters with several input clips: algorithmic bytes = nin reads + 1 write per sample"""
    if skip(name):
        return
    clips = [vz.DeviceClip(fmt, w, h, frames) for _ in range(nin + 1)]
    for i, c in enumerate(clips[:nin]):
        c.fill_noise(1234 + i)
    if prep:
        prep(clips)
    ms = timed(lambda: run(clips), args.reps)
    record(name, fmt, w, h, frames, (nin + 1) * clips[0].frame_bytes, ms)
    for c in clips:
        c.free()


def stats_cfg(name, fmt, w, h, frames, make_filter):
    if skip(name):
        return
    src = vz.DeviceClip(fmt, w, h, frames)
    src.fill_noise(1234)
    f = make_filter(src)
    lib = vz.load_library()
    import ctypes as C
    # time the kernels only: results stay on the device (out = NULL), the stream is not synchronised per call
    ms = timed(lambda: vz._check(lib.vszip_planeminmax_device(f.handle, src.handle, None, 0, frames, None, st.cuda_stream))
               if isinstance(f, vz.PlaneMinMaxFilter) else
               vz._check(lib.vszip_planeaverage_device(f.handle, src.handle, None, 0, frames, None, st.cuda_stream)), args.reps)
    record(name, fmt, w, h, frames, src.frame_bytes, ms)
    src.free()


N = args.frames
pixel_cfg("C1 BoxBlur(13,1,13,1) comptime path", "YUV420P16", 1920, 1080, N, lambda s: vz.BoxBlurFilter(s.info(), hradius=13, hpasses=1, vradius=13, vpasses=1))
pixel_cfg("C2 BoxBlur(13,5,13,5) runtime path [headline]", "YUV420P16", 1920, 1080, N, lambda s: vz.BoxBlurFilter(s.info(), hradius=13, hpasses=5, vradius=13, vpasses=5))
pixel_cfg("C1 on 8-bit frames (YUV420P8): the fused comptime kernel, byte rows widened on the way in", "YUV420P8", 1920, 1080, N, lambda s: vz.BoxBlurFilter(s.info(), hradius=13, hpasses=1, vradius=13, vpasses=1))
pixel_cfg("C2 on 8-bit frames (YUV420P8): the same segment kernels behind a widen/narrow step", "YUV420P8", 1920, 1080, N, lambda s: vz.BoxBlurFilter(s.info(), hradius=13, hpasses=5, vradius=13, vpasses=5))
pixel_cfg("C2 on constant frames (README BlankClip)", "YUV420P16", 1920, 1080, N, lambda s: vz.BoxBlurFilter(s.info(), hradius=13, hpasses=5, vradius=13, vpasses=5), noise=False)
pixel_cfg("C3 Bilateral(sigmaS=2,sigmaR=2) all planes", "YUV420P16", 1920, 1080, N, lambda s: vz.BilateralFilter(s.info(), sigmaS=2, sigmaR=2, planes=[0, 1, 2]))
pixel_cfg("C3' Bilateral default sigmaR=0.02 (exact smem LUT)", "YUV420P16", 1920, 1080, N, lambda s: vz.BilateralFilter(s.info(), sigmaS=2, sigmaR=0.02, planes=[0, 1, 2]))
pixel_cfg("C3'' Bilateral(sigmaS=8, sigmaR=0.1): PBFIC luma (num=4) + alg 2 chroma", "YUV420P16", 1920, 1080, min(N, 32), lambda s: vz.BilateralFilter(s.info(), sigmaS=8, sigmaR=0.1, planes=[0, 1, 2]))
pixel_cfg("C3'' Bilateral(sigmaS=3, sigmaR=0.02, algorithm=1): PBFIC num=12/13", "YUV420P16", 1920, 1080, min(N, 32), lambda s: vz.BilateralFilter(s.info(), sigmaS=3, sigmaR=0.02, algorithm=1, planes=[0, 1, 2]))
pixel_cfg("C6 Limiter(tv_range=True) (pointwise neighbour, 8f rank 3)", "YUV420P16", 1920, 1080, N, lambda s: vz.LimiterFilter(s.info(), tv_range=True))
_lf = {}
multi_cfg("C7 LimitFilter(flt, src, dark_thr=8, bright_thr=8, elast=3) (8f rank 3)", "YUV420P16", 1920, 1080, N, 2,
          lambda c: _lf.setdefault("a", vz.LimitFilterFilter(c[0].info(), c[0].info(), None, dark_thr=8, bright_thr=8, elast=3)).run_device(c[0], c[1], c[2], count=N, stream=st.cuda_stream))
multi_cfg("C7 LimitFilter(flt, src, ref, ...) three inputs", "YUV420P16", 1920, 1080, N, 3,
          lambda c: _lf.setdefault("b", vz.LimitFilterFilter(c[0].info(), c[0].info(), c[0].info(), dark_thr=8, bright_thr=8, elast=3)).run_device(c[0], c[1], c[3], ref=c[2], count=N, stream=st.cuda_stream))
def _smooth_noise(dst):
    """noise smoothed by BoxBlur(13, 3 passes): image-like gradients"""
    tmp = vz.DeviceClip(dst.format, dst.width, dst.height, dst.num_frames)
    tmp.fill_noise(99)
    vz.BoxBlurFilter(tmp.info(), hradius=13, hpasses=3, vradius=13, vpasses=3).run_device(tmp, dst, stream=st.cuda_stream)
    torch.cuda.synchronize()
    tmp.free()


def _image_like(c):
    """src = noise smoothed by BoxBlur(13, 3 passes) (image-like gradients), flt = BoxBlur(src, 2), ref = BoxBlur(src, 4):
    the reference's own LimitFilter usage (tests/test_int_parity.py:158-167)"""
    _smooth_noise(c[1])                                                                                                         # src
    vz.BoxBlurFilter(c[1].info(), hradius=2, vradius=2).run_device(c[1], c[0], stream=st.cuda_stream)                           # flt
    if len(c) > 3:
        vz.BoxBlurFilter(c[1].info(), hradius=4, vradius=4).run_device(c[1], c[2], stream=st.cuda_stream)                       # ref
    torch.cuda.synchronize()


multi_cfg("C7' LimitFilter(flt=BoxBlur(src,2), src, dark_thr=1, bright_thr=1, elast=2) image-like content", "YUV420P16", 1920, 1080, N, 2,
          lambda c: _lf.setdefault("d", vz.LimitFilterFilter(c[0].info(), c[0].info(), None, dark_thr=1, bright_thr=1, elast=2)).run_device(c[0], c[1], c[2], count=N, stream=st.cuda_stream), _image_like)
multi_cfg("C7' LimitFilter(flt, src, ref=BoxBlur(src,4), ...) image-like content", "YUV420P16", 1920, 1080, N, 3,
          lambda c: _lf.setdefault("e", vz.LimitFilterFilter(c[0].info(), c[0].info(), c[0].info(), dark_thr=1, bright_thr=1, elast=2)).run_device(c[0], c[1], c[3], ref=c[2], count=N, stream=st.cuda_stream), _image_like)
multi_cfg("C8 AdaptiveBinarize(clip, clip2, c=3) YUV420P8 (8f rank 3)", "YUV420P8", 1920, 1080, N, 2,
          lambda c: _lf.setdefault("c", vz.AdaptiveBinarizeFilter(c[0].info(), c[0].info(), c=3)).run_device(c[0], c[1], c[2], count=N, stream=st.cuda_stream))
M = max(8, N // 2)
stats_cfg("C4 PlaneMinMax(minthr=.1,maxthr=.1) GRAY16 4K", "GRAY16", 3840, 2160, M, lambda s: vz.PlaneMinMaxFilter(s.info(), minthr=0.1, maxthr=0.1))
stats_cfg("C4 PlaneMinMax(minthr=.1,maxthr=.1) GRAYS 4K", "GRAYS", 3840, 2160, M, lambda s: vz.PlaneMinMaxFilter(s.info(), minthr=0.1, maxthr=0.1))
stats_cfg("C4 PlaneMinMax(minthr=.1,maxthr=.1) GRAY8 4K", "GRAY8", 3840, 2160, M, lambda s: vz.PlaneMinMaxFilter(s.info(), minthr=0.1, maxthr=0.1))
stats_cfg("C4 PlaneMinMax no threshold GRAY16 4K", "GRAY16", 3840, 2160, M, lambda s: vz.PlaneMinMaxFilter(s.info()))
stats_cfg("C4 PlaneAverage(exclude=[0,32768]) GRAY16 4K", "GRAY16", 3840, 2160, M, lambda s: vz.PlaneAverageFilter(s.info(), exclude=[0, 32768]))
stats_cfg("C4 PlaneAverage(exclude=[0,1]) GRAYS 4K", "GRAYS", 3840, 2160, M, lambda s: vz.PlaneAverageFilter(s.info(), exclude=[0, 1]))
def both_stats_cfg(fmt, w, h, frames, mm_args, excl):
    """config 4 runs PlaneMinMax and PlaneAverage over the same plane: the two batch calls back to back (two HBM reads)"""
    if skip(f"C4 both {fmt}"):
        return
    src = vz.DeviceClip(fmt, w, h, frames)
    src.fill_noise(1234)
    mmf, avf = vz.PlaneMinMaxFilter(src.info(), **mm_args), vz.PlaneAverageFilter(src.info(), exclude=excl)
    lib = vz.load_library()

    def separate():
        vz._check(lib.vszip_planeminmax_device(mmf.handle, src.handle, None, 0, frames, None, st.cuda_stream))
        vz._check(lib.vszip_planeaverage_device(avf.handle, src.handle, None, 0, frames, None, st.cuda_stream))
    record(f"C4 PlaneMinMax(thr)+PlaneAverage {fmt} 4K, both batch calls back to back", fmt, w, h, frames, src.frame_bytes, timed(separate, args.reps))
    _, fused = vz.plane_stats_device(mmf, avf, src, count=frames, stream=st.cuda_stream, fetch=False)
    ms = timed(lambda: vz.plane_stats_device(mmf, avf, src, count=frames, stream=st.cuda_stream, fetch=False), args.reps)
    record(f"C4 vszip_planestats_device {fmt} 4K ({'ONE read, fused kernel' if fused else 'not eligible: two reads'}) (8f rank 4)", fmt, w, h, frames, src.frame_bytes, ms)
    src.free()


both_stats_cfg("GRAY16", 3840, 2160, M, dict(minthr=0.1, maxthr=0.1), [0, 32768])
both_stats_cfg("GRAYS", 3840, 2160, M, dict(minthr=0.1, maxthr=0.1), [0, 1])
K = max(4, N // 16)
pixel_cfg("C5a BoxBlur(13,1,13,1) YUV444PS 4K (comptime float)", "YUV444PS", 3840, 2160, K, lambda s: vz.BoxBlurFilter(s.info(), hradius=13, vradius=13))
pixel_cfg("C5b Bilateral(2,2) YUV444PS 4K", "YUV444PS", 3840, 2160, K, lambda s: vz.BilateralFilter(s.info(), sigmaS=2, sigmaR=2))


def _cv2_clahe(job):
    import cv2
    cv2.setNumThreads(1)
    planes, limit, tiles = job
    c = cv2.createCLAHE(limit, tiles)
    return [c.apply(p) for p in planes]


def clahe_cfgs():
    """Device-resident batches (frames/s, read-once-write-once GB/s), get_frame on pinned host frames from 8 threads, and OpenCV's
    CPU CLAHE on the same frames over every host core (one frame per worker, one OpenCV thread per worker) for comparison."""
    import ctypes as C
    import multiprocessing
    import os
    import time
    from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

    lib = vz.load_library()
    for fmt, w, h in (("YUV420P8", 1920, 1080), ("YUV420P16", 1920, 1080), ("GRAY16", 3840, 2160)):
        frames = N if fmt == "YUV420P8" else max(8, N // 4)
        for content in ("noise", "image-like"):
            tag = f"clahe {fmt} {w}x{h} {content}"
            if skip(tag):
                continue
            src, dst = vz.DeviceClip(fmt, w, h, frames), vz.DeviceClip(fmt, w, h, frames)
            if content == "noise":
                src.fill_noise(1234)
            else:
                _smooth_noise(src)
            host = [src.download(i) for i in range(4)]
            for tiles in ([3, 3], [8, 8]):
                f = vz.CLAHEFilter(src.info(), limit=15, tiles=tiles)
                ms = timed(lambda: f.run_device(src, dst, first=0, count=frames, stream=st.cuda_stream), args.reps)
                record(f"{tag} limit=15 tiles={tiles} device batch", fmt, w, h, frames, 2 * src.frame_bytes, ms)
                # get_frame: page-locked host planes, 8 requests in flight on one handle
                def pinned(a):
                    t = torch.empty(a.nbytes, dtype=torch.uint8, pin_memory=True)
                    return t.numpy().view(a.dtype).reshape(a.shape), t
                ins = [[pinned(p) for p in fr] for fr in host]
                for fr, pf in zip(host, ins):
                    for p, (q, _) in zip(fr, pf):
                        q[...] = p
                outs = [[pinned(p) for p in fr] for fr in host for _ in range(2)]
                def one(i):
                    s = vz._cframe([q for q, _ in ins[i % 4]])
                    d = vz._cframe([q for q, _ in outs[i % 8]])
                    vz._check(lib.vszip_clahe_get_frame(f.handle, i, C.byref(s), C.byref(d)))
                n_e2e = 4 * frames
                with ThreadPoolExecutor(8) as ex:
                    list(ex.map(one, range(16)))
                    t0 = time.perf_counter()
                    list(ex.map(one, range(n_e2e)))
                    e2e = time.perf_counter() - t0
                record(f"{tag} limit=15 tiles={tiles} get_frame, pinned frames, 8 threads (end to end)", fmt, w, h, n_e2e,
                       2 * src.frame_bytes, e2e * 1e3)
                workers = os.cpu_count() or 1
                n_cpu = 2 * workers
                with ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("fork")) as ex:
                    list(ex.map(_cv2_clahe, [(host[0], 15.0, tuple(tiles))] * workers))
                    t0 = time.perf_counter()
                    list(ex.map(_cv2_clahe, [(host[i % 4], 15.0, tuple(tiles)) for i in range(n_cpu)]))
                    cpu = time.perf_counter() - t0
                record(f"{tag} limit=15 tiles={tiles} OpenCV 4.13, not the reference: cv2.createCLAHE on {workers} host cores",
                       fmt, w, h, n_cpu, 2 * src.frame_bytes, cpu * 1e3)
            src.free(); dst.free()


clahe_cfgs()


def _cv2_colormap(job):
    import cv2
    cv2.setNumThreads(1)
    y, color = job
    return cv2.applyColorMap(y, color)


def colormap_cfgs():
    """ColorMap: device-resident batches (frames/s; algorithmic bytes = the luma read + 3 * w * h written), get_frame on pinned host
    frames from 8 threads, and OpenCV's applyColorMap on 8-bit luma over every host core (one frame per worker, one OpenCV thread per
    worker) for comparison.  Each batch (1 GB and more) is larger than the L2."""
    import ctypes as C
    import multiprocessing
    import os
    import time
    from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

    lib = vz.load_library()
    for fmt, w, h in (("GRAY8", 1920, 1080), ("GRAY16", 3840, 2160)):
        tag = f"colormap {fmt} {w}x{h} noise"
        if skip(tag):
            continue
        frames = N if fmt == "GRAY8" else max(8, N // 4)
        src, dst = vz.DeviceClip(fmt, w, h, frames), vz.DeviceClip("RGB24", w, h, frames)
        src.fill_noise(1234)
        algo = src.frame_bytes + 3 * w * h
        f = vz.ColorMapFilter(src.info(), 20)
        ms = timed(lambda: f.run_device(src, dst, first=0, count=frames, stream=st.cuda_stream), args.reps)
        record(f"{tag} device batch", fmt, w, h, frames, algo, ms)
        host = [src.download(i) for i in range(4)]

        def pinned(shape, dtype):
            t = torch.empty(int(np.prod(shape)) * np.dtype(dtype).itemsize, dtype=torch.uint8, pin_memory=True)
            return t.numpy().view(dtype).reshape(shape), t
        ins = [pinned(fr[0].shape, fr[0].dtype) for fr in host]
        for (q, _), fr in zip(ins, host):
            q[...] = fr[0]
        outs = [[pinned((h, w), np.uint8) for _ in range(3)] for _ in range(8)]

        def one(i):
            s = vz._cframe([ins[i % 4][0]])
            d = vz._cframe([q for q, _ in outs[i % 8]])
            vz._check(lib.vszip_colormap_get_frame(f.handle, i, C.byref(s), C.byref(d)))
        n_e2e = 4 * frames
        with ThreadPoolExecutor(8) as ex:
            list(ex.map(one, range(16)))
            t0 = time.perf_counter()
            list(ex.map(one, range(n_e2e)))
            e2e = time.perf_counter() - t0
        record(f"{tag} get_frame, pinned frames, 8 threads (end to end)", fmt, w, h, n_e2e, algo, e2e * 1e3)
        if fmt == "GRAY8":
            workers = os.cpu_count() or 1
            n_cpu = 8 * workers
            with ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("fork")) as ex:
                list(ex.map(_cv2_colormap, [(host[0][0], 20)] * workers))
                t0 = time.perf_counter()
                list(ex.map(_cv2_colormap, [(host[i % 4][0], 20) for i in range(n_cpu)], chunksize=4))
                cpu = time.perf_counter() - t0
            record(f"{tag} OpenCV 4.13: cv2.applyColorMap on {workers} host cores", fmt, w, h, n_cpu, algo, cpu * 1e3)
        src.free(); dst.free()


colormap_cfgs()


def _np_packrgb(job):
    r, g, b, bits = job
    u = lambda p: np.minimum(p.astype(np.uint32), 1023) if bits == 10 else p.astype(np.uint32)
    top, sh = (0xC0000000, 10) if bits == 10 else (0xFF000000, 8)
    return np.uint32(top) | u(r) << np.uint32(2 * sh) | u(g) << np.uint32(sh) | u(b)


def packrgb_cfgs():
    """PackRGB: device-resident batches (frames/s; algorithmic bytes = the three planes read + 4 * w * h written), get_frame on pinned
    host frames from 8 threads, and the same pack in numpy over every host core (one frame per worker) for comparison.  Each batch
    (1.8 GB and more) is larger than the L2."""
    import ctypes as C
    import multiprocessing
    import os
    import time
    from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

    lib = vz.load_library()
    for fmt, w, h in (("RGB24", 1920, 1080), ("RGB30", 3840, 2160)):
        tag = f"packrgb {fmt} {w}x{h} noise"
        if skip(tag):
            continue
        frames = N if fmt == "RGB24" else max(8, N // 4)
        src, dst = vz.DeviceClip(fmt, w, h, frames), vz.DeviceClip("GRAY32", w, h, frames)
        src.fill_noise(1234)
        algo = src.frame_bytes + 4 * w * h
        f = vz.PackRGBFilter(src.info())
        ms = timed(lambda: f.run_device(src, dst, first=0, count=frames, stream=st.cuda_stream), args.reps)
        record(f"{tag} device batch", fmt, w, h, frames, algo, ms)
        host = [src.download(i) for i in range(4)]

        def pinned(shape, dtype):
            t = torch.empty(int(np.prod(shape)) * np.dtype(dtype).itemsize, dtype=torch.uint8, pin_memory=True)
            return t.numpy().view(dtype).reshape(shape), t
        ins = [[pinned(p.shape, p.dtype) for p in fr] for fr in host]
        for fr, pf in zip(host, ins):
            for p, (q, _) in zip(fr, pf):
                q[...] = p
        outs = [pinned((h, w), np.uint32) for _ in range(8)]

        def one(i):
            s = vz._cframe([q for q, _ in ins[i % 4]])
            d = vz._cframe([outs[i % 8][0]])
            vz._check(lib.vszip_packrgb_get_frame(f.handle, i, C.byref(s), C.byref(d)))
        n_e2e = 4 * frames
        with ThreadPoolExecutor(8) as ex:
            list(ex.map(one, range(16)))
            t0 = time.perf_counter()
            list(ex.map(one, range(n_e2e)))
            e2e = time.perf_counter() - t0
        record(f"{tag} get_frame, pinned frames, 8 threads (end to end)", fmt, w, h, n_e2e, algo, e2e * 1e3)
        workers = os.cpu_count() or 1
        n_cpu = 2 * workers
        bits = vz.FORMATS[fmt].bits_per_sample
        with ProcessPoolExecutor(workers, mp_context=multiprocessing.get_context("fork")) as ex:
            list(ex.map(_np_packrgb, [(*host[0], bits)] * workers))
            t0 = time.perf_counter()
            list(ex.map(_np_packrgb, [(*host[i % 4], bits) for i in range(n_cpu)]))
            cpu = time.perf_counter() - t0
        record(f"{tag} numpy pack on {workers} host cores", fmt, w, h, n_cpu, algo, cpu * 1e3)
        src.free(); dst.free()


packrgb_cfgs()


def _gpu():
    """the card the numbers were measured on, read in the same run"""
    import subprocess
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


out = {"peak_GBps": PEAK, "gpu": _gpu(), "results": results}
print(json.dumps(out))
if args.out:
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
