"""PlaneMinMax / PlaneAverage parity on the GPU against the CPU oracle and the reference's goldens.
Integer results (min, max, integer average numerators) are exact; float averages and diffs are
f64 tree sums compared at 1e-12 relative (the reference sums sequentially in f64)."""
import json
from pathlib import Path

import numpy as np
import pytest

import oracle_api as oa
import vapoursynth_zip_b200 as vz
from helpers import noise_clip, to_node
from oracle import fixtures as fx

pytestmark = pytest.mark.gpu
GOLD_MM = json.loads((Path(__file__).resolve().parent / "golden" / "planeminmax.json").read_text())
GOLD_AV = json.loads((Path(__file__).resolve().parent / "golden" / "planeaverage.json").read_text())


def props_close(got, want, rel=1e-12):
    assert set(got) == set(want), (got, want)
    for k, w in want.items():
        g = got[k]
        gl, wl = (g, w) if isinstance(w, list) else ([g], [w])
        assert len(gl) == len(wl), (k, g, w)
        for a, b in zip(gl, wl):
            if isinstance(b, int):
                assert a == b, (k, g, w)
            else:
                assert a == pytest.approx(b, rel=rel, abs=1e-300), (k, g, w)


def mm(clip, clipb=None, **args):
    node = to_node(clip).vszip.PlaneMinMax(clipb=to_node(clipb) if clipb is not None else None, **args)
    return node.get_frame(0).props


def av(clip, clipb=None, **args):
    node = to_node(clip).vszip.PlaneAverage(clipb=to_node(clipb) if clipb is not None else None, **args)
    return node.get_frame(0).props


@pytest.mark.parametrize("key", sorted(GOLD_MM))
def test_planeminmax_golden(key):
    fmt, geo, args, variant = oa.parse_case_id(key)
    clip = fx.make_clip(fmt, geo)
    clipb = None
    if bool(args.pop("variant_clipb", 0)) or variant == "ref":
        clipb = oa.boxblur(clip, hradius=1, vradius=1)
    got = mm(clip, clipb, **args)
    want = oa.planeminmax(clip, clipb=clipb, **args)
    props_close(got, want)
    prop = args.get("prop", "psm")
    golden = {prop + k: v for k, v in GOLD_MM[key].items()}
    props_close(got, golden, rel=1e-9)


@pytest.mark.parametrize("key", sorted(k for k in GOLD_AV if "|ref" not in k))
def test_planeaverage_golden(key):
    fmt, geo, args, variant = oa.parse_case_id(key)
    clip = fx.make_clip(fmt, geo)
    got = av(clip, **args)
    props_close(got, oa.planeaverage(clip, **args))
    prop = args.get("prop", "psm")
    props_close({prop + "Avg": got[prop + "Avg"]}, {prop + "Avg": GOLD_AV[key]["avg"]}, rel=1e-9)


@pytest.mark.parametrize("exact", ["0", "1"])
@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY10", "GRAY16", "GRAYH", "GRAYS", "YUV420P16", "RGBS"])
def test_noise_planeminmax(fmt, exact, monkeypatch):
    # exact=1 forces the two-pass radix select; 0 lets the sampled single-read path resolve what it can
    monkeypatch.setenv("VSZIP_MINMAX_EXACT", exact)
    base = "GRAY16" if fmt == "GRAY10" else fmt
    clip = noise_clip(base, 517, 243, seed=9)
    if fmt == "GRAY10":
        clip = {"format": "GRAY10", "planes": [clip["planes"][0] >> 6]}
    other = noise_clip(base, 517, 243, seed=10)
    if fmt == "GRAY10":
        other = {"format": "GRAY10", "planes": [other["planes"][0] >> 6]}
    planes = list(range(len(clip["planes"])))
    for thr in ((0, 0), (0.1, 0.1), (0.4, 0.0), (0.0, 0.33), (0.5, 0.5), (1.0, 1.0), (0.999, 0.001)):
        for b in (None, other):
            args = dict(minthr=thr[0], maxthr=thr[1], planes=planes)
            props_close(mm(clip, b, **args), oa.planeminmax(clip, clipb=b, **args))


@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY16", "GRAYH", "GRAYS", "YUV420P8", "YUV444PS"])
def test_noise_planeaverage(fmt):
    clip = noise_clip(fmt, 517, 243, seed=19)
    other = noise_clip(fmt, 517, 243, seed=20)
    planes = list(range(len(clip["planes"])))
    for ex in ([-1], [0], [128], [100, 150, 200], [0, 1]):
        for b in (None, other):
            props_close(av(clip, b, exclude=ex, planes=planes), oa.planeaverage(clip, ex, clipb=b, planes=planes))


def test_threshold_drop_semantics():
    """tests/test_planeminmax.py:99-110 of the reference."""
    z = np.zeros((8, 64), np.uint8)
    r = np.full((24, 64), 200, np.uint8)
    src = vz.core.clip_from_frames("GRAY8", [[np.vstack([z, r])]])
    assert src.vszip.PlaneMinMax(minthr=0.2).get_frame(0).props["psmMin"] == 0
    assert src.vszip.PlaneMinMax(minthr=0.3).get_frame(0).props["psmMin"] == 200
    src2 = vz.core.clip_from_frames("GRAY8", [[np.vstack([np.full((24, 64), 100, np.uint8), np.full((8, 64), 255, np.uint8)])]])
    assert src2.vszip.PlaneMinMax(maxthr=0.2).get_frame(0).props["psmMax"] == 255
    assert src2.vszip.PlaneMinMax(maxthr=0.3).get_frame(0).props["psmMax"] == 100


def test_blank_clips_and_prop_rename():
    """tests/test_planeminmax.py:147-160, :227-236 and tests/test_planeaverage.py:138-147 of the reference."""
    src = vz.core.BlankClip("YUV420P16", 64, 32, color=[6777, 32768, 0])
    out = src.vszip.PlaneMinMax(minthr=0.2, maxthr=0.3)
    out = out.vszip.PlaneMinMax(minthr=0.2, maxthr=0.3, prop="mm_test")
    p = out.get_frame(0).props
    assert p["psmMin"] == p["mm_testMin"] == 6777 and p["psmMax"] == p["mm_testMax"] == 6777
    h = vz.core.BlankClip("GRAYH", 64, 32, color=0.5).vszip.PlaneMinMax().get_frame(0).props
    assert h["psmMin"] == 0.5 and h["psmMax"] == 0.5
    g = vz.core.BlankClip("GRAY16", 64, 64, color=30000)
    assert g.vszip.PlaneMinMax(minthr=1.0).get_frame(0).props["psmMin"] == 65535
    assert g.vszip.PlaneMinMax(maxthr=1.0).get_frame(0).props["psmMax"] == 0
    a = src.vszip.PlaneAverage(exclude=[300, 5000])
    a = a.vszip.PlaneAverage(exclude=[300, 5000], prop="avg_test")
    p = a.get_frame(0).props
    assert p["psmAvg"] == 0.10341039139391164 and p["avg_testAvg"] == p["psmAvg"]
    multi = src.vszip.PlaneAverage(exclude=[-1], planes=[0, 1, 2]).get_frame(0).props["psmAvg"]
    assert multi == [6777 / 65535, 32768 / 65535, 0.0]


def test_long_exclude_lists():
    """Lists beyond the 16 entries carried in the kernel arguments (the reference takes any length)."""
    rng = np.random.default_rng(5)
    for fmt in ("GRAY8", "GRAY16", "GRAYS"):
        clip = noise_clip(fmt, 317, 143, seed=41)
        other = noise_clip(fmt, 317, 143, seed=42)
        if fmt == "GRAYS":  # float clips compare against f32(int): make some samples hit
            clip["planes"][0][::3, ::2] = 1.0
            clip["planes"][0][1::5, 1::4] = 0.0
        for n in (17, 40, 200):
            ex = [int(v) for v in rng.integers(0, 256 if fmt != "GRAY16" else 65536, n)] + [0, 1]
            props_close(av(clip, exclude=ex), oa.planeaverage(clip, ex))
            props_close(av(clip, other, exclude=ex), oa.planeaverage(clip, ex, clipb=other))


def test_exclude_duplicates_and_out_of_range_values():
    """The packed 16-bit path removes excluded samples arithmetically, so duplicates must be folded and values
    outside the sample range ignored (planeaverage.zig:120-139 compares u16 == i32)."""
    clip = noise_clip("GRAY16", 333, 77, seed=8)
    clip["planes"][0][::2, ::3] = 5
    clip["planes"][0][1::4, 1::5] = 65535
    for ex in ([5, 5, 70000, 5], [65535, -7, 65535, 5, 5], [1, 2, 3, 4, 5], [1, 2, 3, 4, 5, 5, 4], [-1, 65536]):
        props_close(av(clip, exclude=ex), oa.planeaverage(clip, ex))
    ten = {"format": "GRAY10", "planes": [(clip["planes"][0] >> 6).astype(np.uint16)]}
    props_close(av(ten, exclude=[0, 1023, 77]), oa.planeaverage(ten, [0, 1023, 77]))


def test_exclude_exact():
    """tests/test_planeaverage.py:118-128 of the reference."""
    two = np.vstack([np.full((32, 64), 1000, np.uint16), np.full((32, 64), 3000, np.uint16)])
    src = vz.core.clip_from_frames("GRAY16", [[two]])
    assert src.vszip.PlaneAverage(exclude=[1000]).get_frame(0).props["psmAvg"] == 3000 / 65535
    assert src.vszip.PlaneAverage(exclude=[3000]).get_frame(0).props["psmAvg"] == 1000 / 65535
    assert src.vszip.PlaneAverage(exclude=[1000, 3000]).get_frame(0).props["psmAvg"] == 0.0
    twof = np.vstack([np.full((32, 64), 3.0, np.float32), np.full((32, 64), 1.0, np.float32)])
    assert vz.core.clip_from_frames("GRAYS", [[twof]]).vszip.PlaneAverage(exclude=[3]).get_frame(0).props["psmAvg"] == 1.0


def _structured(kind, w, h, rng):
    y, x = np.mgrid[0:h, 0:w]
    if kind == "gradient":
        return ((x * 65535) // (w - 1)).astype(np.uint16)
    if kind == "dark_noise":      # fade-to-black: everything within a few codes of 4096
        return (4096 + rng.integers(-2, 3, (h, w))).astype(np.uint16)
    if kind == "letterbox":       # flat bars hold the min rank, picture holds the max rank
        img = rng.integers(8000, 60000, (h, w)).astype(np.uint16)
        img[: h // 6] = 4096
        img[-(h // 6):] = 4096
        return img
    if kind == "sparse":          # 8-bit content shifted to 16 bits: only every 256th code is used
        return (rng.integers(0, 256, (h, w)) << 8).astype(np.uint16)
    if kind == "rows":            # the row sample misrepresents the plane: rare rows carry the extremes
        img = np.full((h, w), 30000, np.uint16)
        img[1::16] = rng.integers(0, 65536, (len(range(1, h, 16)), w)).astype(np.uint16)
        return img
    if kind == "ten_bit_invalid":  # GRAY10 with samples above the peak (skipped by the reference)
        img = rng.integers(0, 1024, (h, w)).astype(np.uint16)
        img[::7, ::5] = 40000
        return img
    raise KeyError(kind)


@pytest.mark.parametrize("kind", ["gradient", "dark_noise", "letterbox", "sparse", "rows", "ten_bit_invalid"])
def test_structured_planeminmax(kind):
    """Content on which the sampled brackets are wide, degenerate or wrong: results must stay exact."""
    rng = np.random.default_rng(77)
    fmt = "GRAY10" if kind == "ten_bit_invalid" else "GRAY16"
    for (w, h) in ((640, 480), (1283, 721)):
        clip = {"format": fmt, "planes": [_structured(kind, w, h, rng)]}
        for thr in ((0.1, 0.1), (0.02, 0.4), (0.3, 0.0), (0.0005, 0.0005)):
            args = dict(minthr=thr[0], maxthr=thr[1])
            props_close(mm(clip, **args), oa.planeminmax(clip, **args))


def _edge_content(kind, dtype, peak, w, h, rng):
    """Planes whose requested ranks fall at the ends of the sample range, where the bracket windows of the single-read kernel
    (2^k - 1 bins, never starting at bin 0) are clamped or lose bin 0."""
    n = w * h
    if kind == "mostly_zero":      # min rank in bin 0, max rank just above it
        img = np.zeros(n, np.float64)
        idx = rng.choice(n, n // 20, replace=False)
        img[idx] = rng.integers(1, 6, idx.size)
    elif kind == "all_zero":
        img = np.zeros(n, np.float64)
    elif kind == "mostly_peak":    # max rank in the top bin, min rank a few bins below it
        img = np.full(n, peak, np.float64)
        idx = rng.choice(n, n // 20, replace=False)
        img[idx] = peak - rng.integers(1, 6, idx.size)
    elif kind == "both_ends":      # a third at 0, a third at the peak, the rest spread out
        img = rng.integers(0, int(peak) + 1, n).astype(np.float64)
        img[rng.random(n) < 0.33] = 0
        img[rng.random(n) < 0.33] = peak
    elif kind == "low_codes":      # everything inside the first 40 codes: both windows are clamped at bin 1
        img = rng.integers(0, 40, n).astype(np.float64)
    else:
        raise KeyError(kind)
    img = img.reshape(h, w)
    if np.issubdtype(dtype, np.floating):
        return (img / peak).astype(dtype)
    return img.astype(dtype)


@pytest.mark.parametrize("kind", ["mostly_zero", "all_zero", "mostly_peak", "both_ends", "low_codes"])
@pytest.mark.parametrize("fmt", ["GRAY8", "GRAY10", "GRAY16", "GRAYS"])
def test_planeminmax_ranks_at_the_ends_of_the_range(fmt, kind):
    rng = np.random.default_rng(5)
    dtype, peak = {"GRAY8": (np.uint8, 255), "GRAY10": (np.uint16, 1023), "GRAY16": (np.uint16, 65535), "GRAYS": (np.float32, 65535)}[fmt]
    for (w, h) in ((333, 207), (1283, 900)):   # sampled completely / by lines
        clip = {"format": fmt, "planes": [_edge_content(kind, dtype, peak, w, h, rng)]}
        for thr in ((0.1, 0.1), (0.001, 0.6), (0.7, 0.02), (0.04, 0.04)):
            args = dict(minthr=thr[0], maxthr=thr[1])
            props_close(mm(clip, **args), oa.planeminmax(clip, **args))


@pytest.mark.parametrize("fmt", ["GRAY16", "GRAYS"])
def test_full_size_config4(fmt):
    """BASELINE config 4: 3840x2160 GRAY16 / GRAYS, PlaneMinMax(minthr, maxthr) + PlaneAverage(exclude)."""
    clip = noise_clip(fmt, 3840, 2160, seed=31)
    args = dict(minthr=0.1, maxthr=0.1)
    props_close(mm(clip, **args), oa.planeminmax(clip, **args))
    ex = [0, 32768] if fmt == "GRAY16" else [0, 1]
    props_close(av(clip, exclude=ex), oa.planeaverage(clip, ex))
    # a constant plane: every sample in one bin (the reference README's BlankClip case)
    const = vz.core.BlankClip(fmt, 3840, 2160, color=0.25 if fmt == "GRAYS" else 12345)
    p = const.vszip.PlaneMinMax(**args).get_frame(0).props
    want = oa.planeminmax({"format": fmt, "planes": const.get_frame(0).planes}, **args)
    props_close(p, want)


def test_device_batch():
    fmt, w, h, n = "GRAY16", 640, 360, 4
    a, b = vz.DeviceClip(fmt, w, h, n), vz.DeviceClip(fmt, w, h, n)
    a.fill_noise(seed=1)
    b.fill_noise(seed=2)
    mmf = vz.PlaneMinMaxFilter(a.info(), b.info(), minthr=0.1, maxthr=0.2)
    avf = vz.PlaneAverageFilter(a.info(), b.info(), exclude=[7, 9])
    got_mm = mmf.run_device(a, b)
    got_av = avf.run_device(a, b)
    for i in range(n):
        ca = {"format": fmt, "planes": a.download(i)}
        cb = {"format": fmt, "planes": b.download(i)}
        props_close(got_mm[i], oa.planeminmax(ca, minthr=0.1, maxthr=0.2, clipb=cb))
        props_close(got_av[i], oa.planeaverage(ca, [7, 9], clipb=cb))


def test_device_batch_frame_limit():
    """One call takes at most 32768 frames: above that the pair is not fused, and the separate PlaneMinMax call reports the limit."""
    a = vz.DeviceClip("GRAY8", 16, 16, 32769)
    mmf = vz.PlaneMinMaxFilter(a.info(), None, minthr=0.1, maxthr=0.1)
    avf = vz.PlaneAverageFilter(a.info(), None, exclude=[3])
    with pytest.raises(vz.Error, match="^PlaneMinMax: batches above 32768 frames are not supported$"):
        mmf.run_device(a)
    with pytest.raises(vz.Error, match="^PlaneAverage: batches above 32768 frames are not supported$"):
        avf.run_device(a)
    with pytest.raises(vz.Error, match="^PlaneMinMax: batches above 32768 frames are not supported$"):
        vz.plane_stats_device(mmf, avf, a)


def test_minmax_exact_env_and_the_pair(monkeypatch):
    """VSZIP_MINMAX_EXACT=1, read on every call, turns off the sampled threshold path that the fused pair needs; PlaneMinMax without
    thresholds is still fused.  Either way the props equal the separate calls."""
    fmt, w, h, n = "GRAY16", 640, 360, 3
    a = vz.DeviceClip(fmt, w, h, n)
    a.fill_noise(seed=5)
    avf = vz.PlaneAverageFilter(a.info(), None, exclude=[7])
    for exact, mm_args, want_fused in (("1", dict(minthr=0.1, maxthr=0.2), False), ("1", dict(), True), ("0", dict(minthr=0.1, maxthr=0.2), True)):
        monkeypatch.setenv("VSZIP_MINMAX_EXACT", exact)
        mmf = vz.PlaneMinMaxFilter(a.info(), None, **mm_args)
        got, fused = vz.plane_stats_device(mmf, avf, a)
        assert fused == want_fused, (exact, mm_args)
        sep_mm, sep_av = mmf.run_device(a), avf.run_device(a)
        for i in range(n):
            want = dict(sep_mm[i]); want.update(sep_av[i])
            assert got[i] == want, (exact, mm_args, i)



@pytest.mark.parametrize(("fmt", "w", "h", "n"), [("GRAY16", 1920, 1080, 5), ("YUV420P16", 640, 360, 4), ("GRAY10", 517, 243, 3), ("GRAYS", 640, 360, 2), ("GRAYS", 3840, 2160, 2), ("GRAY8", 517, 243, 2)])
def test_minmax_and_average_from_one_read(fmt, w, h, n):
    """SURVEY 8f rank 4: vszip_planestats_device - one kernel reads each plane once and yields both filters' props when the pair is
    eligible (integer and float clips, with and without thresholds; see the rule below); equal to the separate calls and the oracle."""
    base = "GRAY16" if fmt == "GRAY10" else fmt
    a = vz.DeviceClip(fmt, w, h, n)
    if fmt == "GRAY10":
        src = [noise_clip(base, w, h, seed=40 + i)["planes"][0] >> 6 for i in range(n)]
        for i, p in enumerate(src):
            a.upload(i, [p])
    else:
        a.fill_noise(seed=21)
    planes = [0, 1, 2] if fmt.startswith("YUV") else [0]
    is_float = fmt == "GRAYS"
    top = 255 if fmt == "GRAY8" else 65535   # the sample storage decides which exclude values can ever match
    if fmt == "GRAY8":
        a.upload(0, [np.full((h, w), 200, np.uint8)])   # a flat frame next to the noise frames
    cases = [(dict(minthr=0.1, maxthr=0.2), [0, 32768]), (dict(minthr=0.1, maxthr=0.2), [200, 7, 255]), (dict(minthr=0.1, maxthr=0.2), []), (dict(minthr=0.05, maxthr=0.3), [7]),
             (dict(minthr=0.1, maxthr=0.0), [1, 2, 3, 4]), (dict(minthr=0.2, maxthr=0.1), [70000, -1, 5, 5, 9]),
             (dict(minthr=0.1, maxthr=0.2), [1, 2, 3, 4, 5]), (dict(), [0, 1]), (dict(), [3, 1, 4, 1, 5, 9, 2, 6]), (dict(), list(range(17)))]
    for mm_args, excl in cases:
        if is_float:
            excl = [e for e in excl if 0 <= e <= 1] or [0]
        # eligible: no thresholds and <= 16 exclude values, or thresholds and <= 4 distinct values that can match a sample
        distinct = set(excl) if is_float else {e for e in excl if 0 <= e <= top}
        want_fused = (len(excl) <= 16) if not mm_args else len(distinct) <= 4
        mmf = vz.PlaneMinMaxFilter(a.info(), None, planes=planes, **mm_args)
        avf = vz.PlaneAverageFilter(a.info(), None, exclude=excl, planes=planes)
        sep_mm, sep_av = mmf.run_device(a), avf.run_device(a)
        got, fused = vz.plane_stats_device(mmf, avf, a)
        assert fused == want_fused, (fmt, mm_args, excl, fused)
        for i in range(n):
            want = dict(sep_mm[i]); want.update(sep_av[i])
            props_close(got[i], want)
            if fused and (not is_float or not mm_args):
                # integer sums are exact, and without thresholds the float sum is accumulated in the same order as the separate call;
                # the bracket kernel cuts the plane differently, so a float average may differ from the separate call in the last bits
                assert got[i] == want, (fmt, mm_args, excl, i)
        ca = {"format": fmt, "planes": a.download(n - 1)}
        props_close({k: v for k, v in got[n - 1].items() if k in ("psmMin", "psmMax")}, oa.planeminmax(ca, planes=planes, **mm_args))
        props_close({k: v for k, v in got[n - 1].items() if k == "psmAvg"}, oa.planeaverage(ca, excl, planes=planes))
    # different plane sets are not fused; a sub-range of the clip
    if fmt == "YUV420P16":
        mmf = vz.PlaneMinMaxFilter(a.info(), None, planes=[0], minthr=0.1, maxthr=0.1)
        avf = vz.PlaneAverageFilter(a.info(), None, exclude=[3], planes=[0, 1])
        got, fused = vz.plane_stats_device(mmf, avf, a, first=1, count=2)
        assert not fused and len(got) == 2 and got[1]["psmMax"] == mmf.run_device(a)[2]["psmMax"] and got[0]["psmAvg"] == avf.run_device(a)[1]["psmAvg"]
