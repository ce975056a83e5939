"""vapoursynth_zip_b200 — Python host mirror of the vszip plugin surface for the B200 hot path.

The product is the C-ABI library (include/vszip_cuda.h, built into lib/libvszip_cuda.so from
csrc/*.cu).  This module is the thin host side used where the reference would be driven through
VapourSynth: it mirrors the `clip.vszip.BoxBlur / Bilateral / PlaneMinMax / PlaneAverage / ... / CLAHE / ColorMap` call
surface (same names, arguments, defaults, frame props and error messages; src/vszip.zig:46-69,
:184-199) on top of a minimal clip/frame model, so the parity tests read like the reference's own
tests (tests/test_boxblur.py etc. of the reference).  All arithmetic happens in the CUDA library;
there is no CPU fallback and a missing library or GPU raises `Error`.
"""
from __future__ import annotations

import ctypes as C
import weakref
import os
from dataclasses import dataclass
from pathlib import Path

import numpy as np

__all__ = ["Error", "core", "plane_stats_device", "VideoFormat", "VideoFrame", "VideoNode", "DeviceClip", "GRAY", "RGB", "YUV", "INTEGER", "FLOAT"]

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("VSZIP_CUDA_LIB") or (_PKG / "lib" / "libvszip_cuda.so"))  # override: A/B builds only

GRAY, RGB, YUV = 1, 2, 3          # VapourSynth4.h VSColorFamily
INTEGER, FLOAT = 0, 1             # VSSampleType


class Error(RuntimeError):
    """Mirror of vapoursynth.Error: raised with the reference's message on invalid arguments."""


# --------------------------------------------------------------------------- ctypes structs
class _VideoInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("width", "height", "num_frames", "color_family", "sample_type", "bits_per_sample",
                                         "bytes_per_sample", "sub_sampling_w", "sub_sampling_h", "num_planes")]


class _Frame(C.Structure):
    _fields_ = [("data", C.c_void_p * 3), ("stride", C.c_ssize_t * 3)]


class _BoxBlurArgs(C.Structure):
    _fields_ = [("planes", C.POINTER(C.c_int64)), ("num_planes", C.c_int32),
                ("has_hradius", C.c_int32), ("hradius", C.c_int64), ("has_hpasses", C.c_int32), ("hpasses", C.c_int64),
                ("has_vradius", C.c_int32), ("vradius", C.c_int64), ("has_vpasses", C.c_int32), ("vpasses", C.c_int64)]


class _BilateralArgs(C.Structure):
    _fields_ = [("sigmaS", C.POINTER(C.c_double)), ("num_sigmaS", C.c_int32), ("sigmaR", C.POINTER(C.c_double)), ("num_sigmaR", C.c_int32),
                ("planes", C.POINTER(C.c_int64)), ("num_planes", C.c_int32), ("algorithm", C.POINTER(C.c_int64)), ("num_algorithm", C.c_int32),
                ("PBFICnum", C.POINTER(C.c_int64)), ("num_PBFICnum", C.c_int32)]


class _BilateralInfo(C.Structure):
    _fields_ = [("sigmaS", C.c_double * 3), ("sigmaR", C.c_double * 3), ("process", C.c_int32 * 3), ("algorithm", C.c_int32 * 3),
                ("PBFICnum", C.c_uint32 * 3), ("radius", C.c_uint32 * 3), ("samples", C.c_uint32 * 3), ("step", C.c_uint32 * 3),
                ("exact_lut", C.c_int32 * 3)]


class _MinMaxArgs(C.Structure):
    _fields_ = [("has_minthr", C.c_int32), ("minthr", C.c_double), ("has_maxthr", C.c_int32), ("maxthr", C.c_double),
                ("planes", C.POINTER(C.c_int64)), ("num_planes", C.c_int32)]


class _MinMaxProps(C.Structure):
    _fields_ = [("count", C.c_int32), ("plane", C.c_int32 * 3), ("is_float", C.c_int32), ("has_diff", C.c_int32),
                ("imin", C.c_int64 * 3), ("imax", C.c_int64 * 3), ("fmin", C.c_double * 3), ("fmax", C.c_double * 3), ("diff", C.c_double * 3)]


class _AverageArgs(C.Structure):
    _fields_ = [("exclude", C.POINTER(C.c_int64)), ("num_exclude", C.c_int32), ("planes", C.POINTER(C.c_int64)), ("num_planes", C.c_int32)]


class _LimiterArgs(C.Structure):
    _fields_ = [("min", C.POINTER(C.c_double)), ("num_min", C.c_int32), ("max", C.POINTER(C.c_double)), ("num_max", C.c_int32),
                ("planes", C.POINTER(C.c_int64)), ("num_planes", C.c_int32), ("has_tv_range", C.c_int32), ("tv_range", C.c_int32),
                ("has_mask", C.c_int32), ("mask", C.c_int32)]


class _LimitFilterArgs(C.Structure):
    _fields_ = [("dark_thr", C.POINTER(C.c_double)), ("num_dark_thr", C.c_int32), ("bright_thr", C.POINTER(C.c_double)), ("num_bright_thr", C.c_int32),
                ("elast", C.POINTER(C.c_double)), ("num_elast", C.c_int32), ("planes", C.POINTER(C.c_int64)), ("num_planes", C.c_int32),
                ("color_range", C.c_int32)]


class _AdaptiveBinarizeArgs(C.Structure):
    _fields_ = [("has_c", C.c_int32), ("c", C.c_int64)]


class _ClaheArgs(C.Structure):
    _fields_ = [("has_limit", C.c_int32), ("limit", C.c_double), ("tiles", C.POINTER(C.c_int64)), ("num_tiles", C.c_int32)]


class _ColorMapArgs(C.Structure):
    _fields_ = [("has_color", C.c_int32), ("color", C.c_int64)]


class _AverageProps(C.Structure):
    _fields_ = [("count", C.c_int32), ("plane", C.c_int32 * 3), ("has_diff", C.c_int32), ("avg", C.c_double * 3), ("diff", C.c_double * 3)]


# every symbol include/vszip_cuda.h declares: (restype, argtypes)
_P = C.c_void_p
ABI = {
    "vszip_cuda_init": (C.c_int, [C.POINTER(C.c_int32), C.c_int32]),
    "vszip_cuda_shutdown": (None, []),
    "vszip_cuda_device_count": (C.c_int, []),
    "vszip_cuda_last_error": (C.c_char_p, []),
    "vszip_cuda_abi_version": (C.c_int, []),
    "vszip_cuda_kernel_launches": (C.c_uint64, []),
    "vszip_cuda_transfer_bytes": (C.c_uint64, [C.c_int32]),
    "vszip_cuda_stream_sync": (C.c_int, [C.c_int32, _P]),
    "vszip_cuda_host_forget": (None, [_P]),
    "vszip_cuda_host_registered_bytes": (C.c_size_t, []),
    "vszip_cuda_host_register_limit": (C.c_size_t, [C.c_size_t]),
    "vszip_cuda_reserve": (C.c_int32, [C.POINTER(_VideoInfo), C.c_int32]),
    "vszip_boxblur_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_BoxBlurArgs)]),
    "vszip_boxblur_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_boxblur_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_bilateral_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_VideoInfo), C.POINTER(_BilateralArgs)]),
    "vszip_bilateral_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_bilateral_get_info": (C.c_int, [_P, C.POINTER(_BilateralInfo)]),
    "vszip_bilateral_device": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_planeminmax_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_VideoInfo), C.POINTER(_MinMaxArgs)]),
    "vszip_planeminmax_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_MinMaxProps)]),
    "vszip_planeminmax_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.POINTER(_MinMaxProps), _P]),
    "vszip_planeaverage_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_VideoInfo), C.POINTER(_AverageArgs)]),
    "vszip_planeaverage_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_AverageProps)]),
    "vszip_planeaverage_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.POINTER(_AverageProps), _P]),
    "vszip_planestats_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.POINTER(_MinMaxProps), C.POINTER(_AverageProps), C.POINTER(C.c_int32), _P]),
    "vszip_planestats_device_b": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, C.POINTER(_MinMaxProps), C.POINTER(_AverageProps),
                                            C.POINTER(C.c_int32), _P]),
    "vszip_filter_free": (None, [_P]),
    "vszip_filter_planes": (C.c_int, [_P, C.POINTER(C.c_int32 * 3)]),
    "vszip_dev_clip_alloc": (_P, [C.POINTER(_VideoInfo), C.c_int32, C.c_int32]),
    "vszip_dev_clip_free": (None, [_P]),
    "vszip_dev_clip_upload": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame)]),
    "vszip_dev_clip_download": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame)]),
    "vszip_dev_clip_fill_noise": (C.c_int, [_P, C.c_uint64, C.c_int32, C.c_int32]),
    "vszip_dev_clip_frame_bytes": (C.c_size_t, [_P]),
    "vszip_dev_clip_plane_ptr": (_P, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_ssize_t)]),
    "vszip_limiter_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_LimiterArgs)]),
    "vszip_limiter_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_limiter_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_limitfilter_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_VideoInfo), C.POINTER(_VideoInfo), C.POINTER(_LimitFilterArgs)]),
    "vszip_limitfilter_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_limitfilter_get_info": (C.c_int, [_P, C.POINTER(C.c_float * 3), C.POINTER(C.c_float * 3), C.POINTER(C.c_float * 3)]),
    "vszip_limitfilter_device": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_adaptivebinarize_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_VideoInfo), C.POINTER(_AdaptiveBinarizeArgs)]),
    "vszip_adaptivebinarize_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_adaptivebinarize_device": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_clahe_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_ClaheArgs)]),
    "vszip_clahe_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_clahe_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_colormap_create": (_P, [C.POINTER(_VideoInfo), C.POINTER(_ColorMapArgs)]),
    "vszip_colormap_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame)]),
    "vszip_colormap_device": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P]),
    "vszip_colormap_get_lut": (C.c_int, [_P, C.POINTER(C.c_uint8 * 768)]),
    "vszip_filter_output_info": (C.c_int, [_P, C.POINTER(_VideoInfo)]),
    "vszip_chain_create": (_P, [C.POINTER(_P), C.c_int32]),
    "vszip_chain_create2": (_P, [C.POINTER(_P), C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "vszip_chain_free": (None, [_P]),
    "vszip_chain_planes": (C.c_int, [_P, C.POINTER(C.c_int32 * 3)]),
    "vszip_chain_get_frame": (C.c_int, [_P, C.c_int32, C.POINTER(_Frame), C.POINTER(_Frame), C.POINTER(_P)]),
}

_lib = None


def load_library():
    """dlopen the C-ABI library and bind every declared symbol.  Fails loudly if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise Error(f"{LIB_PATH} is missing: build the CUDA extension with `make` (or __graft_entry__.build()); "
                    "vapoursynth_zip_b200 has no CPU fallback")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in ABI.items():
        fn = getattr(lib, name)  # AttributeError = ABI mismatch between header and library
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _last_error() -> str:
    return (load_library().vszip_cuda_last_error() or b"").decode("utf-8", "replace")


# --------------------------------------------------------------------------- formats
@dataclass(frozen=True)
class VideoFormat:
    name: str
    color_family: int
    sample_type: int
    bits_per_sample: int
    bytes_per_sample: int
    subsampling_w: int
    subsampling_h: int
    num_planes: int

    @property
    def dtype(self):
        if self.sample_type == FLOAT:
            return {2: np.float16, 4: np.float32}[self.bytes_per_sample]
        return {1: np.uint8, 2: np.uint16, 4: np.uint32}[self.bytes_per_sample]

    def plane_shape(self, width, height, plane):
        sw, sh = (self.subsampling_w, self.subsampling_h) if plane else (0, 0)
        return (height >> sh, width >> sw)


def _mk(name, fam, st, bits, ssw=0, ssh=0):
    bps = 1 if bits <= 8 else (2 if bits <= 16 else 4)
    return VideoFormat(name, fam, st, bits, bps, ssw, ssh, 1 if fam == GRAY else 3)


FORMATS = {f.name: f for f in [
    _mk("GRAY8", GRAY, INTEGER, 8), _mk("GRAY9", GRAY, INTEGER, 9), _mk("GRAY10", GRAY, INTEGER, 10), _mk("GRAY11", GRAY, INTEGER, 11),
    _mk("GRAY12", GRAY, INTEGER, 12), _mk("GRAY14", GRAY, INTEGER, 14), _mk("GRAY16", GRAY, INTEGER, 16),
    _mk("GRAY32", GRAY, INTEGER, 32), _mk("GRAYH", GRAY, FLOAT, 16), _mk("GRAYS", GRAY, FLOAT, 32),
    _mk("YUV420P8", YUV, INTEGER, 8, 1, 1), _mk("YUV420P10", YUV, INTEGER, 10, 1, 1), _mk("YUV420P16", YUV, INTEGER, 16, 1, 1),
    _mk("YUV420PH", YUV, FLOAT, 16, 1, 1), _mk("YUV420PS", YUV, FLOAT, 32, 1, 1),
    _mk("YUV422P16", YUV, INTEGER, 16, 1, 0),
    _mk("YUV444P8", YUV, INTEGER, 8), _mk("YUV444P10", YUV, INTEGER, 10), _mk("YUV444P16", YUV, INTEGER, 16),
    _mk("YUV444PH", YUV, FLOAT, 16), _mk("YUV444PS", YUV, FLOAT, 32),
    _mk("RGB24", RGB, INTEGER, 8), _mk("RGB30", RGB, INTEGER, 10), _mk("RGB48", RGB, INTEGER, 16),
    _mk("RGBH", RGB, FLOAT, 16), _mk("RGBS", RGB, FLOAT, 32),
]}
globals().update(FORMATS)  # vz.GRAY16, vz.YUV420P16, ... like the vs.* presets


def _fmt(f) -> VideoFormat:
    return f if isinstance(f, VideoFormat) else FORMATS[f]


def _format_of(vi: _VideoInfo) -> VideoFormat:
    """The preset with this video info's format."""
    key = (vi.color_family, vi.sample_type, vi.bits_per_sample, vi.bytes_per_sample, vi.sub_sampling_w, vi.sub_sampling_h, vi.num_planes)
    for f in FORMATS.values():
        if (f.color_family, f.sample_type, f.bits_per_sample, f.bytes_per_sample, f.subsampling_w, f.subsampling_h, f.num_planes) == key:
            return f
    raise Error(f"no format preset for {key}")


def _vi(fmt: VideoFormat, width, height, num_frames) -> _VideoInfo:
    return _VideoInfo(width, height, num_frames, fmt.color_family, fmt.sample_type, fmt.bits_per_sample, fmt.bytes_per_sample,
                      fmt.subsampling_w, fmt.subsampling_h, fmt.num_planes)


def _rows(p):
    """Planes are passed with their own row stride; only the samples of a row must be contiguous."""
    return p if (p.ndim == 2 and p.strides[1] == p.itemsize and p.strides[0] > 0) else np.ascontiguousarray(p)


def _cframe(planes) -> _Frame:
    fr = _Frame()
    fr._keep = list(planes)  # the struct only holds raw pointers: keep the arrays alive with it
    for i, p in enumerate(planes):
        if p is None:
            continue
        assert p.ndim == 2 and p.strides[1] == p.itemsize, "plane rows must be contiguous"
        fr.data[i] = p.ctypes.data
        fr.stride[i] = p.strides[0]
    return fr


# --------------------------------------------------------------------------- clip model
class VideoFrame:
    def __init__(self, fmt: VideoFormat, width: int, height: int, planes, props=None):
        self.format, self.width, self.height = fmt, width, height
        self.planes = list(planes)
        self.props = dict(props or {})

    def __getitem__(self, plane):
        return self.planes[plane]

    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


class VideoNode:
    """A clip: format + geometry + a frame getter.  `clip.vszip.X(...)` mirrors the plugin namespace."""

    _op = None  # a vszip node's _Op

    def __init__(self, fmt: VideoFormat, width: int, height: int, num_frames: int, getter):
        self.format, self.width, self.height, self.num_frames = fmt, width, height, num_frames
        self._getter = getter

    def get_frame(self, n: int) -> VideoFrame:
        if not 0 <= n < self.num_frames:
            raise Error(f"frame {n} out of range")
        chain = _fusable_chain(self) if core.fuse_chains else None
        if chain is not None:
            return _fused_get(chain, n)
        return self._getter(n)

    @property
    def vszip(self):
        return _Namespace(self)

    def _info(self) -> _VideoInfo:
        return _vi(self.format, self.width, self.height, self.num_frames)


def _i64(values):
    vals = [int(v) for v in values]
    return (C.c_int64 * max(len(vals), 1))(*vals), len(vals)


def _f64(values):
    vals = [float(v) for v in values]
    return (C.c_double * max(len(vals), 1))(*vals), len(vals)


def _as_list(v):
    if v is None:
        return None
    return list(v) if isinstance(v, (list, tuple, np.ndarray)) else [v]


_live_filters = weakref.WeakSet()


class _Filter:
    """Owns one vszip_filter handle.  Each filter class states how its kind runs, like the library's KindInfo table:
    GET_FRAME is its `vszip_*_get_frame` symbol; ARGS lists that entry point's frame arguments by the chain's numbering of the
    clips (0 = the main input, 1 = the second clip, 2 = the third), and the first of them is the clip whose frame gives the output
    its untouched planes and its props; PROPS is the props struct a stats filter fills (None: the filter has a pixel output), DROP
    the props it rewrites, without their prefix."""

    GET_FRAME, ARGS, PROPS, DROP = None, (0,), None, ()

    def __init__(self, handle, node: VideoNode | None = None):
        if not handle:
            raise Error(_last_error())
        self.handle = handle
        mask = (C.c_int32 * 3)()
        load_library().vszip_filter_planes(handle, C.byref(mask))
        self.process = [bool(m) for m in mask]  # the planes it reads
        self.out_info = _VideoInfo()            # the format of the frames it returns
        _check(load_library().vszip_filter_output_info(handle, C.byref(self.out_info)))
        _live_filters.add(self)

    def _device(self, fn, clips, first, count, stream, prop=None):
        """One `vszip_*_device` call on `clips`, in its argument order (None: an optional clip left out), for `count` frames from
        `first` (default: the rest of the first clip).  A stats filter returns its props, one dict per frame."""
        count = clips[0].num_frames - first if count is None else count
        handles = [c.handle if c else None for c in clips]
        if self.PROPS is None:
            _check(fn(self.handle, *handles, first, count, stream))
            return None
        out = (self.PROPS * max(count, 1))()
        _check(fn(self.handle, *handles, first, count, out, stream))
        return _props_list(self.to_props, out, count, prop)

    def close(self):
        """vszip_filter_free (xxxFree in the reference's glue); also called by core.shutdown() for every instance still alive."""
        h, self.handle = getattr(self, "handle", None), None
        if h and _lib is not None:
            _lib.vszip_filter_free(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _check(rc):
    if rc != 0:
        raise Error(_last_error())


def _planes_arg(planes):
    if planes is None:
        return None, -1
    return _i64(_as_list(planes))


# ---- BoxBlur
class BoxBlurFilter(_Filter):
    GET_FRAME = "vszip_boxblur_get_frame"

    def __init__(self, vi: _VideoInfo, planes=None, hradius=None, hpasses=None, vradius=None, vpasses=None):
        pl, npl = _planes_arg(planes)
        a = _BoxBlurArgs(pl, npl, hradius is not None, int(hradius or 0), hpasses is not None, int(hpasses or 0),
                         vradius is not None, int(vradius or 0), vpasses is not None, int(vpasses or 0))
        super().__init__(load_library().vszip_boxblur_create(C.byref(vi), C.byref(a)))

    def run_device(self, src: "DeviceClip", dst: "DeviceClip", first=0, count=None, stream=None):
        self._device(load_library().vszip_boxblur_device, (src, dst), first, count, stream)


class BilateralFilter(_Filter):
    GET_FRAME, ARGS = "vszip_bilateral_get_frame", (0, 1)

    def __init__(self, vi: _VideoInfo, ref_vi: _VideoInfo | None = None, sigmaS=None, sigmaR=None, planes=None, algorithm=None, PBFICnum=None):
        s, ns = _f64(_as_list(sigmaS) or [])
        r, nr = _f64(_as_list(sigmaR) or [])
        al, na = _i64(_as_list(algorithm) or [])
        pb, npb = _i64(_as_list(PBFICnum) or [])
        pl, npl = _planes_arg(planes)
        a = _BilateralArgs(s, ns, r, nr, pl, npl, al, na, pb, npb)
        super().__init__(load_library().vszip_bilateral_create(C.byref(vi), C.byref(ref_vi) if ref_vi is not None else None, C.byref(a)))

    def info(self):
        out = _BilateralInfo()
        _check(load_library().vszip_bilateral_get_info(self.handle, C.byref(out)))
        return out

    def run_device(self, src, dst, ref=None, first=0, count=None, stream=None):
        self._device(load_library().vszip_bilateral_device, (src, ref, dst), first, count, stream)


def _props_from(prop, keys, count, getter):
    """Append semantics (src/vapoursynth/planeminmax.zig:48-72): scalar for one plane, list for several."""
    out = {}
    for key in keys:
        vals = [getter(key, i) for i in range(count)]
        out[prop + key] = vals[0] if len(vals) == 1 else vals
    return out


def _props_list(to_props, arr, count, prop):
    """The props of `count` frames from an array of props structs."""
    return [to_props(arr[i], prop) for i in range(count)]


class PlaneMinMaxFilter(_Filter):
    GET_FRAME, ARGS, PROPS, DROP = "vszip_planeminmax_get_frame", (0, 1), _MinMaxProps, ("Diff", "Max", "Min")

    def __init__(self, vi: _VideoInfo, clipb_vi: _VideoInfo | None = None, minthr=None, maxthr=None, planes=None):
        pl, npl = _planes_arg(planes)
        a = _MinMaxArgs(minthr is not None, float(minthr or 0), maxthr is not None, float(maxthr or 0), pl, npl)
        super().__init__(load_library().vszip_planeminmax_create(C.byref(vi), C.byref(clipb_vi) if clipb_vi is not None else None, C.byref(a)))

    @staticmethod
    def to_props(p: _MinMaxProps, prop="psm"):
        if p.count == 0:
            return {}
        def get(key, i):
            if key == "Diff":
                return p.diff[i]
            if p.is_float:
                return p.fmin[i] if key == "Min" else p.fmax[i]
            return int(p.imin[i]) if key == "Min" else int(p.imax[i])
        return _props_from(prop, ("Min", "Max") + (("Diff",) if p.has_diff else ()), p.count, get)

    def run_device(self, clipa, clipb=None, first=0, count=None, stream=None, prop="psm"):
        return self._device(load_library().vszip_planeminmax_device, (clipa, clipb), first, count, stream, prop)


class PlaneAverageFilter(_Filter):
    GET_FRAME, ARGS, PROPS, DROP = "vszip_planeaverage_get_frame", (0, 1), _AverageProps, ("Diff", "Avg")

    def __init__(self, vi: _VideoInfo, clipb_vi: _VideoInfo | None = None, exclude=None, planes=None):
        pl, npl = _planes_arg(planes)
        if exclude is None:
            ex, nex = None, -1
        else:
            ex, nex = _i64(_as_list(exclude))
        a = _AverageArgs(ex, nex, pl, npl)
        super().__init__(load_library().vszip_planeaverage_create(C.byref(vi), C.byref(clipb_vi) if clipb_vi is not None else None, C.byref(a)))

    @staticmethod
    def to_props(p: _AverageProps, prop="psm"):
        if p.count == 0:
            return {}
        out = _props_from(prop, ("Avg",), p.count, lambda k, i: p.avg[i])
        if p.has_diff:
            out.update(_props_from(prop, ("Diff",), p.count, lambda k, i: p.diff[i]))
        return out

    def run_device(self, clipa, clipb=None, first=0, count=None, stream=None, prop="psm"):
        return self._device(load_library().vszip_planeaverage_device, (clipa, clipb), first, count, stream, prop)


def plane_stats_device(minmax: "PlaneMinMaxFilter", average: "PlaneAverageFilter", clipa, first=0, count=None, stream=None, prop="psm", fetch=True,
                       clipb=None):
    """PlaneMinMax + PlaneAverage over the same device-resident frames (vszip_planestats_device, or vszip_planestats_device_b with
    clipb): one read of each plane (pair) when the pair is eligible.  Returns (props per frame - both filters' props merged, like
    `clip.vszip.PlaneMinMax().vszip.PlaneAverage()` -, fused)."""
    count = clipa.num_frames - first if count is None else count
    mm = (_MinMaxProps * max(count, 1))() if fetch else None
    av = (_AverageProps * max(count, 1))() if fetch else None
    fused = C.c_int32(0)
    if clipb is None:
        _check(load_library().vszip_planestats_device(minmax.handle, average.handle, clipa.handle, first, count, mm, av, C.byref(fused), stream))
    else:
        _check(load_library().vszip_planestats_device_b(minmax.handle, average.handle, clipa.handle, clipb.handle, first, count, mm, av,
                                                        C.byref(fused), stream))
    if not fetch:
        return None, bool(fused.value)
    out = _props_list(PlaneMinMaxFilter.to_props, mm, count, prop)
    for p, q in zip(out, _props_list(PlaneAverageFilter.to_props, av, count, prop)):
        p.update(q)
    return out, bool(fused.value)


class LimiterFilter(_Filter):
    GET_FRAME = "vszip_limiter_get_frame"

    def __init__(self, vi: _VideoInfo, min=None, max=None, tv_range=None, mask=None, planes=None):
        pl, npl = _planes_arg(planes)
        mn, nmn = (None, -1) if min is None else _f64(_as_list(min))
        mx, nmx = (None, -1) if max is None else _f64(_as_list(max))
        a = _LimiterArgs(mn, nmn, mx, nmx, pl, npl, tv_range is not None, int(bool(tv_range)), mask is not None, int(bool(mask)))
        super().__init__(load_library().vszip_limiter_create(C.byref(vi), C.byref(a)))

    def run_device(self, src: "DeviceClip", dst: "DeviceClip", first=0, count=None, stream=None):
        self._device(load_library().vszip_limiter_device, (src, dst), first, count, stream)


class LimitFilterFilter(_Filter):
    """vszip.LimitFilter (src/vapoursynth/limit_filter.zig:93-124).  color_range: the flt clip's _ColorRange (0 full, 1 limited, None absent)."""

    GET_FRAME, ARGS = "vszip_limitfilter_get_frame", (0, 1, 2)

    def __init__(self, flt_vi: _VideoInfo, src_vi: _VideoInfo, ref_vi: _VideoInfo | None = None, dark_thr=None, bright_thr=None, elast=None,
                 planes=None, color_range=None):
        dk, ndk = _f64(_as_list(dark_thr) or [])
        br, nbr = _f64(_as_list(bright_thr) or [])
        el, nel = _f64(_as_list(elast) or [])
        pl, npl = _planes_arg(planes)
        a = _LimitFilterArgs(dk, ndk, br, nbr, el, nel, pl, npl, -1 if color_range is None else int(color_range))
        super().__init__(load_library().vszip_limitfilter_create(C.byref(flt_vi), C.byref(src_vi) if src_vi is not None else None,
                                                                 C.byref(ref_vi) if ref_vi is not None else None, C.byref(a)))

    def info(self):
        d, b, e = (C.c_float * 3)(), (C.c_float * 3)(), (C.c_float * 3)()
        _check(load_library().vszip_limitfilter_get_info(self.handle, C.byref(d), C.byref(b), C.byref(e)))
        return {"dark_thr": list(d), "bright_thr": list(b), "elast": list(e)}

    def run_device(self, flt, src, dst, ref=None, first=0, count=None, stream=None):
        self._device(load_library().vszip_limitfilter_device, (flt, src, ref, dst), first, count, stream)


class AdaptiveBinarizeFilter(_Filter):
    """vszip.AdaptiveBinarize (src/vapoursynth/adaptive_binarize.zig:79-116).  It filters clip2, the chain's main input; the
    output frame is made from clip, which get_frame takes first."""

    GET_FRAME, ARGS = "vszip_adaptivebinarize_get_frame", (1, 0)

    def __init__(self, vi: _VideoInfo, clip2_vi: _VideoInfo, c=None):
        a = _AdaptiveBinarizeArgs(c is not None, int(c or 0))
        super().__init__(load_library().vszip_adaptivebinarize_create(C.byref(vi), C.byref(clip2_vi) if clip2_vi is not None else None, C.byref(a)))

    def run_device(self, clip, clip2, dst, first=0, count=None, stream=None):
        self._device(load_library().vszip_adaptivebinarize_device, (clip, clip2, dst), first, count, stream)


class CLAHEFilter(_Filter):
    """Contrast-limited adaptive histogram equalisation of every plane, bit-exact with OpenCV's CLAHE::apply (DESIGN.md §4.7)."""

    GET_FRAME = "vszip_clahe_get_frame"

    def __init__(self, vi: _VideoInfo, limit=None, tiles=None):
        t, nt = _i64(_as_list(tiles) or [])
        a = _ClaheArgs(limit is not None, float(limit or 0), t, nt)
        super().__init__(load_library().vszip_clahe_create(C.byref(vi), C.byref(a)))

    def run_device(self, src: "DeviceClip", dst: "DeviceClip", first=0, count=None, stream=None):
        self._device(load_library().vszip_clahe_device, (src, dst), first, count, stream)


class ColorMapFilter(_Filter):
    """OpenCV's colormap `color` (cv::ColormapTypes 0..21) on the luma, RGB24 out (DESIGN.md §4.8)."""

    GET_FRAME = "vszip_colormap_get_frame"

    def __init__(self, vi: _VideoInfo, color=None):
        a = _ColorMapArgs(color is not None, int(color or 0))
        super().__init__(load_library().vszip_colormap_create(C.byref(vi), C.byref(a)))

    def lut(self):
        """The selected table as a (256, 3) uint8 array of R, G, B."""
        out = (C.c_uint8 * 768)()
        _check(load_library().vszip_colormap_get_lut(self.handle, C.byref(out)))
        return np.frombuffer(bytes(out), np.uint8).reshape(256, 3).copy()

    def run_device(self, src: "DeviceClip", dst: "DeviceClip", first=0, count=None, stream=None):
        self._device(load_library().vszip_colormap_device, (src, dst), first, count, stream)


class _Namespace:
    """`clip.vszip` / `core.vszip`: the plugin functions with the reference's argument names."""

    def __init__(self, clip: VideoNode | None = None):
        self._clip = clip

    def _c(self, clip):
        clip = clip if clip is not None else self._clip
        if clip is None:
            raise Error("clip argument is required")
        return clip

    def BoxBlur(self, clip=None, planes=None, hradius=None, hpasses=None, vradius=None, vpasses=None) -> VideoNode:
        clip = self._c(clip)
        return _node(BoxBlurFilter(clip._info(), planes, hradius, hpasses, vradius, vpasses), clip)

    def Limiter(self, clip=None, min=None, max=None, tv_range=None, mask=None, planes=None) -> VideoNode:
        clip = self._c(clip)
        return _node(LimiterFilter(clip._info(), min, max, tv_range, mask, planes), clip)

    def CLAHE(self, *pos, **kw) -> VideoNode:
        clip, limit, tiles = self._bind(("clip", "limit", "tiles"), pos, kw)
        if clip is None:
            raise Error("clip argument is required")
        return _node(CLAHEFilter(clip._info(), limit, tiles), clip)

    def ColorMap(self, *pos, **kw) -> VideoNode:
        clip, color = self._bind(("clip", "color"), pos, kw)
        if clip is None:
            raise Error("clip argument is required")
        return _node(ColorMapFilter(clip._info(), color), clip, set_props={"_ColorRange": 0, "_Matrix": 0})

    def _bind(self, names, pos, kw):
        """VapourSynth binding rule: `clip.vszip.F(a, b)` puts the bound clip first and shifts the positional arguments."""
        if self._clip is not None:
            pos = (self._clip,) + tuple(pos)
        if len(pos) > len(names):
            raise Error("too many positional arguments")
        args = dict(zip(names, pos))
        for k, v in kw.items():
            if k not in names:
                raise Error(f"unknown argument {k}")
            if k in args:
                raise Error(f"argument {k} given twice")
            args[k] = v
        return [args.get(k) for k in names]

    def LimitFilter(self, *pos, **kw) -> VideoNode:
        flt, src, ref, dark_thr, bright_thr, elast, planes = self._bind(("flt", "src", "ref", "dark_thr", "bright_thr", "elast", "planes"), pos, kw)
        if flt is None or src is None:
            raise Error("LimitFilter: flt and src are required")
        f = LimitFilterFilter(flt._info(), src._info(), ref._info() if ref is not None else None, dark_thr, bright_thr, elast, planes, None)
        # hz.scaleValue -> hz.getColorRange reads frame 0 of flt (src/helper.zig:259-276), only when the depth is not 8 bits
        if flt.format.bits_per_sample != 8 and flt.num_frames > 0:
            cr = flt.get_frame(0).props.get("_ColorRange")
            if cr is not None:
                f = LimitFilterFilter(flt._info(), src._info(), ref._info() if ref is not None else None, dark_thr, bright_thr, elast, planes, cr)
        return _node(f, flt, src, ref)

    def AdaptiveBinarize(self, *pos, **kw) -> VideoNode:
        clip, clip2, c = self._bind(("clip", "clip2", "c"), pos, kw)
        if clip is None or clip2 is None:
            raise Error("AdaptiveBinarize: clip and clip2 are required")
        f = AdaptiveBinarizeFilter(clip._info(), clip2._info(), c)
        return _node(f, clip2, clip, set_props={"_ColorRange": 0})  # dst_prop.setColorRange(.FULL)

    def Bilateral(self, clip=None, ref=None, sigmaS=None, sigmaR=None, planes=None, algorithm=None, PBFICnum=None) -> VideoNode:
        clip = self._c(clip)
        flt = BilateralFilter(clip._info(), ref._info() if ref is not None else None, sigmaS, sigmaR, planes, algorithm, PBFICnum)
        return _node(flt, clip, ref)

    def PlaneMinMax(self, clipa=None, minthr=None, maxthr=None, clipb=None, planes=None, prop=None) -> VideoNode:
        clipa = self._c(clipa)
        flt = PlaneMinMaxFilter(clipa._info(), clipb._info() if clipb is not None else None, minthr, maxthr, planes)
        return _node(flt, clipa, clipb, prefix="psm" if prop is None else str(prop))

    def PlaneAverage(self, clipa=None, exclude=None, clipb=None, planes=None, prop=None) -> VideoNode:
        clipa = self._c(clipa)
        flt = PlaneAverageFilter(clipa._info(), clipb._info() if clipb is not None else None, exclude, planes)
        return _node(flt, clipa, clipb, prefix="psm" if prop is None else str(prop))


@dataclass(frozen=True)
class _Op:
    """What a vszip node computes: the record its unfused get and the chain planner read."""
    filter: _Filter
    input: VideoNode              # the clip it filters: the chain's input[i]
    second: VideoNode | None      # its second and third clips: the chain's second[i] and third[i]
    third: VideoNode | None
    base: VideoNode               # the clip whose frame gives the output's untouched planes and props
    format: VideoFormat           # the format of the frames it returns: the base clip's unless the filter changes it
    set_props: dict               # props set on every output frame
    prefix: str                   # stats filters: the prefix of the props they write

    def props(self, base_props, stats=None):
        """The output props: the base frame's, minus the stats props this node rewrites, plus the ones it writes and sets."""
        p = dict(base_props)
        if stats is not None:
            for k in self.filter.DROP:
                p.pop(self.prefix + k, None)
            p.update(self.filter.to_props(stats, self.prefix))
        p.update(self.set_props)
        return p

    def get(self, n):
        """Unfused evaluation: the filter's get_frame on frame n of each input; an extra clip that is shorter repeats its last
        frame (rpFrameReuseLastOnly).  Inputs pass their processed planes; a pixel filter's output gets fresh processed planes
        and shares the others with the base frame (newVideoFrame2), or fresh planes of its own format when it changes the format;
        a stats filter's shares every plane (copyFrame)."""
        core._ensure_init()
        flt, clips = self.filter, (self.input, self.second, self.third)
        frames = [None if clips[i] is None else clips[i].get_frame(min(n, clips[i].num_frames - 1)) for i in flt.ARGS]
        base = frames[0]
        args = [None if fr is None else C.byref(_cframe([_rows(p) if flt.process[i] else None for i, p in enumerate(fr.planes)]))
                for fr in frames]
        fmt = self.format
        if flt.PROPS is None and fmt is not base.format:
            planes = [np.empty(fmt.plane_shape(base.width, base.height, i), fmt.dtype) for i in range(fmt.num_planes)]
            stats, out = None, _cframe(planes)
        elif flt.PROPS is None:
            planes = [np.empty_like(p, order="C") if flt.process[i] else p for i, p in enumerate(base.planes)]
            stats, out = None, _cframe([p if flt.process[i] else None for i, p in enumerate(planes)])
        else:
            planes = base.planes
            stats = out = flt.PROPS()
        _check(getattr(load_library(), flt.GET_FRAME)(flt.handle, n, *args, C.byref(out)))
        return VideoFrame(fmt, base.width, base.height, planes, self.props(base.props, stats))


def _node(flt: _Filter, main: VideoNode, second: VideoNode | None = None, third: VideoNode | None = None, set_props=None,
          prefix="") -> VideoNode:
    """A vszip node on `main`, `second` and `third` (the chain's numbering)."""
    base = (main, second, third)[flt.ARGS[0]]
    o, b = flt.out_info, base.format  # the library's output format (vszip_filter_output_info): the base clip's but for ColorMap
    same = (o.color_family, o.sample_type, o.bits_per_sample, o.sub_sampling_w, o.sub_sampling_h, o.num_planes) == (
        b.color_family, b.sample_type, b.bits_per_sample, b.subsampling_w, b.subsampling_h, b.num_planes)
    fmt = b if same else _format_of(o)
    op = _Op(flt, main, second, third, base, fmt, set_props or {}, prefix)
    node = VideoNode(fmt, base.width, base.height, base.num_frames, op.get)
    node.filter, node._op = flt, op
    return node


# ---- fused evaluation of chains of vszip nodes (vszip_chain_*): one upload, one download
class _Chain:
    def __init__(self, nodes, inputs, second, third):
        self.nodes = nodes  # evaluation order
        n = len(nodes)
        handles = (_P * n)(*[nd.filter.handle for nd in nodes])
        arrs = [(C.c_int32 * n)(*v) for v in (inputs, second, third)]
        self.handle = load_library().vszip_chain_create2(handles, n, *arrs)
        if not self.handle:
            raise Error(_last_error())
        w = (C.c_int32 * 3)()
        _check(load_library().vszip_chain_planes(self.handle, C.byref(w)))
        self.written = [bool(v) for v in w]

    def __del__(self):
        try:
            if self.handle and _lib is not None:
                _lib.vszip_chain_free(self.handle)
        except Exception:
            pass
        self.handle = None


def _fusable_chain(node: "VideoNode"):
    """The chain ending in `node` if it and at least one predecessor are vszip nodes whose clips come from inside the chain."""
    cached = getattr(node, "_chain", False)
    if cached is not False:
        return cached
    main, cur = [], node
    while cur._op is not None and len(main) < 16:
        main.append(cur)
        cur = cur._op.input
    node._chain = _plan_chain(main[::-1], cur)
    return node._chain


def _side_input(x, value):
    """A single-input pixel node that is not on the main line but filters a value of the chain (`src.vszip.BoxBlur()` given as
    ref / clipb): it joins the chain right before its reader."""
    op = x._op
    return op is not None and op.filter.PROPS is None and op.second is None and op.third is None and value(op.input) is not None


def _plan_chain(main, source):
    """Elements and value numbers (0 = source, k = output of element k - 1) for vszip_chain_create2.  Walks the main line from the
    source end; a node with an extra clip from outside the chain becomes the source of what follows it."""
    while main:
        elems, vals, cut = [], {id(source): 0}, None
        value = lambda x: vals.get(id(x))
        for k, nd in enumerate(main):
            side = []
            for x in (nd._op.second, nd._op.third):
                if x is None or value(x) is not None or any(x is y for y in side):
                    continue
                if not _side_input(x, value):
                    cut = k
                    break
                side.append(x)
            if cut is not None:
                break
            for x in side + [nd]:
                elems.append(x)
                vals[id(x)] = len(elems) if x._op.filter.PROPS is None else value(x._op.input)  # stats pass their input on
        if cut is not None:
            source, main = main[cut], main[cut + 1:]
        elif len(elems) > 16:
            source, main = main[0], main[1:]
        else:
            break
    if not main or len(elems) < 2:
        return None
    inputs = [value(x._op.input) for x in elems]
    second = [-1 if x._op.second is None else value(x._op.second) for x in elems]
    third = [-1 if x._op.third is None else value(x._op.third) for x in elems]
    return _Chain(elems, inputs, second, third), source


def _fused_get(chain_and_source, n: int) -> "VideoFrame":
    chain, source = chain_and_source
    core._ensure_init()
    src = source.get_frame(n)
    last = chain.nodes[-1]  # the result has the last node's format: the source's, or RGB24 after a ColorMap
    fmt = last.format
    out_planes = [np.empty(fmt.plane_shape(src.width, src.height, i), fmt.dtype) if chain.written[i] else src.planes[i]
                  for i in range(fmt.num_planes)]
    s = _cframe([_rows(p) for p in src.planes])
    d = _cframe([p if chain.written[i] else None for i, p in enumerate(out_planes)])
    outs, ptrs = [], (_P * len(chain.nodes))()
    for i, nd in enumerate(chain.nodes):
        o = None
        if nd._op.filter.PROPS is not None:
            o = nd._op.filter.PROPS()
            ptrs[i] = C.cast(C.pointer(o), _P)
        outs.append(o)
    _check(load_library().vszip_chain_get_frame(chain.handle, n, C.byref(s), C.byref(d), ptrs))
    # every node's props, in evaluation order, exactly as the unfused nodes derive them from the clip their frame comes from
    props = {id(source): src.props}
    for nd, o in zip(chain.nodes, outs):
        props[id(nd)] = nd._op.props(props[id(nd._op.base)], o)
    return VideoFrame(fmt, source.width, source.height, out_planes, props[id(last)])


# --------------------------------------------------------------------------- device-resident clips
class DeviceClip:
    """N frames resident in one GPU's HBM (vszip_dev_clip)."""

    def __init__(self, fmt, width, height, num_frames, device=0):
        core._ensure_init()
        self.format, self.width, self.height, self.num_frames, self.device = _fmt(fmt), width, height, num_frames, device
        vi = _vi(self.format, width, height, num_frames)
        self.handle = load_library().vszip_dev_clip_alloc(C.byref(vi), num_frames, device)
        if not self.handle:
            raise Error(_last_error())

    def info(self) -> _VideoInfo:
        return _vi(self.format, self.width, self.height, self.num_frames)

    @property
    def frame_bytes(self) -> int:
        return int(load_library().vszip_dev_clip_frame_bytes(self.handle))

    def fill_noise(self, seed=1234, first_frame_no=0, frame_no_stride=1):
        _check(load_library().vszip_dev_clip_fill_noise(self.handle, seed, first_frame_no, frame_no_stride))

    def upload(self, frame: int, planes):
        keep = [np.ascontiguousarray(p) for p in planes]
        _check(load_library().vszip_dev_clip_upload(self.handle, frame, C.byref(_cframe(keep))))

    def download(self, frame: int):
        planes = [np.empty(self.format.plane_shape(self.width, self.height, p), self.format.dtype) for p in range(self.format.num_planes)]
        _check(load_library().vszip_dev_clip_download(self.handle, frame, C.byref(_cframe(planes))))
        return planes

    def plane_ptr(self, frame, plane):
        pitch = C.c_ssize_t()
        return load_library().vszip_dev_clip_plane_ptr(self.handle, frame, plane, C.byref(pitch)), pitch.value

    def free(self):
        if self.handle and _lib is not None:
            _lib.vszip_dev_clip_free(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# --------------------------------------------------------------------------- core
class _Core:
    def __init__(self):
        self._ready = False
        # evaluate chains of vszip nodes with one upload and one download (vszip_chain_*)
        self.fuse_chains = os.environ.get("VSZIP_FUSE_CHAINS", "1") != "0"

    def init(self, devices=None) -> int:
        """vszip_cuda_init: `devices` = list of CUDA ordinals (default: all visible, or $VSZIP_CUDA_DEVICES)."""
        lib = load_library()
        if devices is None and os.environ.get("VSZIP_CUDA_DEVICES"):
            devices = [int(x) for x in os.environ["VSZIP_CUDA_DEVICES"].split(",")]
        if devices:
            arr = (C.c_int32 * len(devices))(*devices)
            n = lib.vszip_cuda_init(arr, len(devices))
        else:
            n = lib.vszip_cuda_init(None, 0)
        if n <= 0:
            raise Error(_last_error())
        self._ready = True
        return n

    def reserve(self, info, buffers=2):
        """vszip_cuda_reserve: allocate every request slot's staging buffers for frames of this format now (first-call latency)."""
        self._ensure_init()
        _check(load_library().vszip_cuda_reserve(C.byref(info), buffers))

    def shutdown(self):
        """vszip_cuda_shutdown: frees the per-GPU slots, streams and the host pin cache (filters and clips must be gone)."""
        import gc
        gc.collect()
        for f in list(_live_filters):     # instances the interpreter has not finalised yet: their device tables go first
            f.close()
        load_library().vszip_cuda_shutdown()
        self._ready = False

    def _ensure_init(self):
        if not self._ready:
            self.init()

    @property
    def num_devices(self):
        return load_library().vszip_cuda_device_count()

    @property
    def kernel_launches(self) -> int:
        return int(load_library().vszip_cuda_kernel_launches())

    def transfer_bytes(self, direction=None):
        """vszip_cuda_transfer_bytes: sample bytes of frames copied so far, (host->device, device->host), or one direction (0 / 1)."""
        lib = load_library()
        if direction is not None:
            return int(lib.vszip_cuda_transfer_bytes(direction))
        return int(lib.vszip_cuda_transfer_bytes(0)), int(lib.vszip_cuda_transfer_bytes(1))

    def sync(self, device=0, stream=None):
        _check(load_library().vszip_cuda_stream_sync(device, stream))

    @property
    def vszip(self):
        return _Namespace(None)

    # ---- sources (stand-ins for std.BlankClip / a decoded clip)
    def clip_from_frames(self, fmt, frames, props=None) -> VideoNode:
        """frames: list (one entry per frame) of lists of 2-D numpy planes."""
        fmt = _fmt(fmt)
        h, w = frames[0][0].shape
        for fr in frames:
            assert len(fr) == fmt.num_planes
            for i, p in enumerate(fr):
                assert p.dtype == fmt.dtype and p.shape == fmt.plane_shape(w, h, i), (p.dtype, p.shape, fmt.name)
        return VideoNode(fmt, w, h, len(frames), lambda n: VideoFrame(fmt, w, h, frames[n], props))

    def BlankClip(self, fmt, width, height, length=1, color=None) -> VideoNode:
        fmt = _fmt(fmt)
        color = _as_list(color) or [0] * fmt.num_planes
        color = color + [color[-1]] * (fmt.num_planes - len(color))
        planes = [np.full(fmt.plane_shape(width, height, i), color[i], dtype=fmt.dtype) for i in range(fmt.num_planes)]
        return VideoNode(fmt, width, height, length, lambda n: VideoFrame(fmt, width, height, planes))


core = _Core()
