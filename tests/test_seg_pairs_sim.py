"""The H passes of the segment BoxBlur kernels (csrc/boxblur_seg_core.h: one word per window step holding both of its samples),
replayed lane by lane on the CPU (tests/sim/boxblur_seg_pairs_sim.cpp), against the oracle: bit-exact for every radius the
kernels are instantiated for, on rows that end at a segment end (edge exchange, mirrors from registers), ragged rows (whole
segments republished), one-segment rows and rows barely longer than a window."""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

import oracle

ROOT = Path(__file__).resolve().parents[1]
SIM_SRC = ROOT / "tests" / "sim" / "boxblur_seg_pairs_sim.cpp"
SIM_LIB = ROOT / "build" / "libsegpairsim.so"


@pytest.fixture(scope="module")
def sim():
    SIM_LIB.parent.mkdir(exist_ok=True)
    core = ROOT / "vapoursynth_zip_b200" / "csrc" / "boxblur_seg_core.h"
    if not SIM_LIB.exists() or SIM_LIB.stat().st_mtime < max(SIM_SRC.stat().st_mtime, core.stat().st_mtime):
        subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", f"-I{core.parent}", "-o", str(SIM_LIB), str(SIM_SRC)], check=True)
    lib = C.CDLL(str(SIM_LIB))
    lib.seg_pairs_sim_u16.argtypes = [C.c_int, C.c_void_p, C.c_void_p] + [C.c_int] * 4

    def run(what, src, r, passes=1):
        src = np.ascontiguousarray(src)
        dst = np.zeros_like(src)
        h, w = src.shape
        assert lib.seg_pairs_sim_u16(what, src.ctypes.data, dst.ctypes.data, w, h, r, passes) == 0
        return dst
    return run


def noise(w, h, seed, bits=16):
    return np.random.default_rng(seed).integers(0, 1 << bits, size=(h, w), dtype=np.uint32).astype(np.uint16)


@pytest.mark.parametrize("r", list(range(1, 23)))
def test_h_passes_match_oracle(sim, r):
    for w, passes in ((2 * r + 1, 2), (2 * r + 2, 3), (60, 5), (61, 1), (120, 2), (180, 3), (331, 3), (960, 5), (1920, 4)):
        if w <= 2 * r:
            continue
        src = noise(w, 7, seed=r * 100 + w)
        assert np.array_equal(sim(0, src, r, passes), oracle.boxblur_plane(src, r, passes, 0, 0)), ("H", r, w, passes)


@pytest.mark.parametrize("r", list(range(1, 23)))
def test_comptime_h_pass_matches_oracle(sim, r):
    for w in (2 * r + 1, 61, 120, 331, 960):
        src = noise(w, 5, seed=r * 7 + w)
        assert np.array_equal(sim(1, src, r), oracle.boxblur_plane(src, r, 1, 0, 0)), ("CT H", r, w)


def test_headline_rows(sim):
    """config 2's luma and chroma row lengths, five passes; 10-bit samples too."""
    for w, bits in ((1920, 16), (960, 16), (1920, 10)):
        src = noise(w, 31, seed=w + bits, bits=bits)
        assert np.array_equal(sim(0, src, 13, 5), oracle.boxblur_plane(src, 13, 5, 0, 0))
