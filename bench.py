#!/usr/bin/env python
"""bench.py — BASELINE.json metric on its headline configuration, plus one entry per BASELINE config.

Headline workload (configs[1]): vszip.BoxBlur(hradius=13, hpasses=5, vradius=13, vpasses=5) on 1920x1080 YUV420P16
uniform-noise frames.  One "step" = one pass of that filter over a batch of FRAMES_PER_STEP frames that are already
resident in HBM (`value`) or that live in host memory and go through the getFrame-style C-ABI entry point with both PCIe
copies inside the timed region (`e2e`).

  python bench.py [--gpus N] [--steps K] [--warmup W]          our arm (CUDA, through the C ABI)
  python bench.py --impl reference [...]                       the reference's CPU algorithm (oracle port) on the host cores
  python bench.py --no-configs / --no-cpu                      skip the per-config legs / the cpu_baseline leg
  python bench.py --dump-outputs DIR [...]                     also write a sample of the headline's last-step output to DIR

--steps is the number of timed steps of every GPU leg (headline, H/V split, e2e, configs); the cpu_baseline leg of our
arm is a fixed 8-step sample.  Inputs are generated from fixed seeds, so the same arguments give the same inputs on every run.

The JSON line carries, next to the contract keys:
  configs   one entry per BASELINE.json config (c1..c5): device-resident frames/s, algorithmic GB/s and fraction of the
            measured HBM peak at this N; c5 also end to end through the fused chain frame API
  e2e       value = frames/s through vszip_boxblur_get_frame on frames in pinned host memory (the bench contract's definition);
            `pageable` = the same call on PAGEABLE planes, the way VapourSynth hands them over (library default: CPU copies
            through the slots' pinned staging buffers), `pageable_registered` = the opt-in host pin cache (buffers that come
            back are page-locked in place), `pcie_ceiling_fps` = copy-only probe (same bytes up and down, no kernels) at the same N

Multi-GPU (torchrun, one rank per GPU): frames are independent, every rank processes its own frames (frame n -> GPU n mod k),
no collective on the data path; scaling is weak.  Timed regions are bracketed by barrier + synchronize, timed with CUDA events
on the launching stream (device legs) or the host clock around synchronous calls (e2e legs), max over ranks.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

W, H, FMT = 1920, 1080, "YUV420P16"
ARGS = dict(hradius=13, hpasses=5, vradius=13, vpasses=5)
FRAMES_PER_STEP = 1024
FRAME_BYTES = (W * H + 2 * (W // 2) * (H // 2)) * 2          # 6,220,800 B read per frame
ALGO_BYTES = 2 * FRAME_BYTES                                  # read once + written once (SURVEY 8d)
METRIC = "fps @1080p YUV420P16, vszip.BoxBlur(hradius=13,hpasses=5,vradius=13,vpasses=5), device-resident"
WORKLOAD = "configs[1]: BoxBlur 13/5/13/5 on 1920x1080 YUV420P16 uniform-noise frames"
# identical in both arms (the driver compares it); per-arm batch sizes live under "batch"
CONFIG = {"workload": WORKLOAD, "filter": "vszip.BoxBlur", "args": ARGS, "format": FMT, "width": W, "height": H, "content": "uniform noise",
          "parallelism": "frame-parallel (frame n -> GPU n mod k), no collective",
          "l2": "every timed step streams far more than the 126 MB L2 (inputs larger than L2, no flush needed)"}


DUMP_FRAMES = 4   # 4 whole frames as float32 = 49.8 MB, under the 64 MB a dump may take


def dump_outputs(out_dir, dst, frame_nos):
    """Writes what the headline's last step left in `dst` (what a caller of run_device receives) for comparing two builds:
    DUMP_FRAMES frames of the batch picked with a fixed seed, every plane whole, as float32 (exact for 16-bit samples),
    boxblur_{y,u,v}.npy of shape (DUMP_FRAMES, h, w), and their frame numbers in frame_numbers.npy."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    pick = sorted(np.random.default_rng(0).choice(len(frame_nos), DUMP_FRAMES, replace=False).tolist())
    frames = [dst.download(i) for i in pick]
    for p, name in enumerate("yuv"):
        np.save(out / f"boxblur_{name}.npy", np.stack([f[p] for f in frames]).astype(np.float32))
    np.save(out / "frame_numbers.npy", np.array([frame_nos[i] for i in pick], dtype=np.float64))


def frames_of_rank(rank, world, per_rank):
    """Frame numbers rank `rank` of `world` processes: frame n runs on GPU n mod k (SURVEY 8e)."""
    return [rank + world * i for i in range(per_rank)]


def max_over_ranks(x, world, device=None):
    """Slowest rank's value (the job is as slow as its slowest GPU); works with nccl (cuda) and gloo (cpu)."""
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def cores_of_rank(local, world):
    """Disjoint share of the host cores for this rank's threads (8 ranks x 8 request threads on a 32-core box trample each other)."""
    try:
        allowed = sorted(os.sched_getaffinity(0))
    except AttributeError:
        return None
    per = len(allowed) // max(1, world)
    if world <= 1 or per < 1:
        return allowed
    return allowed[local * per:(local + 1) * per]


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# --------------------------------------------------------------------------- CPU arm (oracle port)
def cpu_arm(steps, warmup, frames_per_step=None):
    """The reference's algorithm on the host cores: one frame per thread, like VapourSynth's fmParallel
    workers (src/vapoursynth/boxblur.zig:211).  The Zig plugin cannot be built in this image (no zig, no
    VapourSynth), so this is the C++ restatement that reproduces the reference's goldens (kind "port")."""
    import numpy as np

    import oracle
    oracle.lib()
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    n = frames_per_step or 2 * cores
    rng = np.random.default_rng(1234)
    frames = [[rng.integers(0, 65536, size=s, dtype=np.uint32).astype(np.uint16) for s in ((H, W), (H // 2, W // 2), (H // 2, W // 2))]
              for _ in range(min(n, 2 * cores))]

    def one(i):
        for p in frames[i % len(frames)]:
            oracle.boxblur_plane(p, ARGS["hradius"], ARGS["hpasses"], ARGS["vradius"], ARGS["vpasses"])

    with ThreadPoolExecutor(cores) as ex:
        for _ in range(warmup):
            list(ex.map(one, range(n)))
        t0 = time.perf_counter()
        for _ in range(steps):
            list(ex.map(one, range(n)))
        dt = time.perf_counter() - t0
    fps = n * steps / dt
    return fps, dt / steps * 1e3, cores, n


CPU_NOTE = ("C++ restatement of vszip 19.0.0 (oracle/), not the Zig binary: written for clarity (per-line heap buffers, column-strided "
            "V pass), so it is slower than the reference's vectorised row-streaming build would be on the same cores")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    fps, ms, cores, n = cpu_arm(steps, warmup)
    sample = f"{n} frames per step ({cores} host threads, one frame per thread), {steps} timed steps after {warmup} warm-up steps"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
        "config": CONFIG, "batch": {"frames_per_step": n, "note": CPU_NOTE},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except FileNotFoundError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        self.p.wait()
        self.f.flush()
        rows = [r.split(",") for r in Path(self.f.name).read_text().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, reasons, mx = [], set(), None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except (ValueError, IndexError):
                continue
            for nm, v in zip(names, r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            # under load = samples in the upper half of what was seen (idle samples before/after the loop drop out)
            hi = sorted(sm)[len(sm) // 2:]
            out.update(sm_mhz=hi[len(hi) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))
        return out


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import vapoursynth_zip_b200 as vz

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    my_cores = cores_of_rank(local, world)
    if my_cores and world > 1:
        os.sched_setaffinity(0, my_cores)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    vz.core.init([local])
    lib = vz.load_library()
    dev = torch.device("cuda", local)
    peak, peak_src = peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ranks(x):
        return max_over_ranks(x, world, dev)

    # launch on a torch-owned stream so torch's CUDA events bracket exactly the kernels (a NULL stream would
    # select the library's own stream, which torch events on the default stream do not see)
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def timed(fn, steps, warmup):
        """ms per step on the launching stream, slowest rank"""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        barrier()
        return max_ranks(ms) / steps

    def timed_host(fn, steps, warmup):
        """seconds per step on the host clock around synchronous calls (the e2e legs), slowest rank"""
        for _ in range(warmup):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        dt = max_ranks(time.perf_counter() - t0)
        barrier()
        return dt / steps

    n = FRAMES_PER_STEP
    src = vz.DeviceClip(FMT, W, H, n, device=0)
    dst = vz.DeviceClip(FMT, W, H, n, device=0)
    mine = frames_of_rank(rank, world, n)                    # frame numbers n with n mod world == rank
    src.fill_noise(seed=1234, first_frame_no=mine[0], frame_no_stride=world)
    flt = vz.BoxBlurFilter(src.info(), **ARGS)

    # ---- headline: device-resident
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = vz.core.kernel_launches
    ms_step = timed(lambda: flt.run_device(src, dst, 0, n, stream), args.steps, args.warmup)
    launches = (vz.core.kernel_launches - l0) * args.steps // (args.steps + args.warmup)
    clocks = sampler.stop() if sampler else None
    fps = world * n / (ms_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dst, mine)   # before the legs below overwrite dst

    # ---- per-kernel durations for the roofline (H passes only / V passes only, same batch)
    fh = vz.BoxBlurFilter(src.info(), hradius=13, hpasses=5, vradius=0, vpasses=0)
    fv = vz.BoxBlurFilter(src.info(), hradius=0, hpasses=0, vradius=13, vpasses=5)
    ms_h = timed(lambda: fh.run_device(src, dst, 0, n, stream), args.steps, 3)
    ms_v = timed(lambda: fv.run_device(src, dst, 0, n, stream), args.steps, 3)
    dom_name, dom_ms = ("hseg_kernel<13> (5 H passes)", ms_h) if ms_h >= ms_v else ("vseg_tile_kernel<13> (5 V passes)", ms_v)
    achieved = ALGO_BYTES * n / (dom_ms * 1e-3) / 1e9
    traffic = None  # DRAM bytes per launch of that kernel, from the committed ncu --set full capture
    tfiles = sorted((ROOT / "profiles").glob("traffic_r*.json"))
    if tfiles:
        per_frame = json.loads(tfiles[-1].read_text())["dram_bytes_per_frame"].get(dom_name.split("<")[0])
        traffic = per_frame * n if per_frame else None
    path_gbs = ALGO_BYTES * n / (ms_step * 1e-3) / 1e9

    # ---- one entry per BASELINE config, device-resident (c5 also end to end), every rank on its own frames
    configs = None if args.no_configs else other_configs(vz, lib, torch, np, timed, timed_host, stream, world, peak, args.steps,
                                                         {"fps": fps, "ms_per_frame_batch": ms_step, "frames": n}, path_gbs, my_cores)
    src.free(); dst.free()

    # ---- end to end: host frames -> vszip_boxblur_get_frame (H2D + kernels + D2H per frame), several requests in flight
    ne = 64
    shapes = [(H, W), (H // 2, W // 2), (H // 2, W // 2)]
    ncores = len(my_cores) if my_cores else 8
    in_flight = max(2, min(8, ncores))           # DMA-bound legs: 8 requests in flight saturate PCIe in both directions
    in_flight_staged = max(2, min(16, ncores))   # memcpy-bound leg: as many worker threads as VapourSynth would run (<= 16 slots per GPU)
    pools = {n: ThreadPoolExecutor(n) for n in {in_flight, in_flight_staged}}
    rng = np.random.default_rng(rank)

    def e2e_leg(frames_in, frames_out, threads):
        pool = pools[threads]
        cin = [vz._cframe(p) for p in frames_in]
        cout = [vz._cframe(p) for p in frames_out]

        def one(i):
            if lib.vszip_boxblur_get_frame(flt.handle, mine[i], C.byref(cin[i]), C.byref(cout[i])):
                raise RuntimeError(vz._last_error())
        s = timed_host(lambda: list(pool.map(one, range(ne))), args.steps, 3)
        return world * ne / s

    # (a) pageable planes, one allocation per plane (anonymous mappings with malloc's 64-byte offset, which is what the
    #     core's aligned allocator returns for buffers of this size), the same buffers coming back every step like
    #     VapourSynth's frame pool: the library's default path, a memcpy through the slots' pinned staging buffers per direction
    import mmap
    maps = []

    def pageable(shape):
        nbytes = int(np.prod(shape)) * 2
        m = mmap.mmap(-1, nbytes + 4096)
        maps.append(m)
        return np.frombuffer(m, dtype=np.uint16, count=nbytes // 2, offset=64).reshape(shape)
    page_in = [[pageable(s) for s in shapes] for _ in range(ne)]
    page_out = [[pageable(s) for s in shapes] for _ in range(ne)]
    for fr in page_in:
        for pl in fr:
            pl[...] = rng.integers(0, 65536, size=pl.shape, dtype=np.uint32).astype(np.uint16)
    lib.vszip_cuda_host_forget(None)
    old_limit = lib.vszip_cuda_host_register_limit(0)
    e2e_staged = e2e_leg(page_in, page_out, in_flight_staged)
    # (b) opt-in: the runtime page-locks a buffer the second time it sees its address and DMAs it in place from then on
    lib.vszip_cuda_host_register_limit(8 << 30)
    e2e_registered = e2e_leg(page_in, page_out, in_flight)
    registered = int(lib.vszip_cuda_host_registered_bytes())
    lib.vszip_cuda_host_forget(None)
    lib.vszip_cuda_host_register_limit(old_limit)
    del page_in, page_out
    maps.clear()
    # (c) application-pinned frames (planes back to back in one pinned allocation per frame)
    host_in = [torch.empty(FRAME_BYTES, dtype=torch.uint8).pin_memory() for _ in range(ne)]
    host_out = [torch.empty(FRAME_BYTES, dtype=torch.uint8).pin_memory() for _ in range(ne)]

    def planes_of(t):
        a = t.numpy().view(np.uint16)
        out, off = [], 0
        for (h, w) in shapes:
            out.append(a[off:off + h * w].reshape(h, w)); off += h * w
        return out

    for t in host_in:
        t.numpy()[:] = rng.integers(0, 256, size=FRAME_BYTES, dtype=np.uint8)
    e2e_pinned = e2e_leg([planes_of(t) for t in host_in], [planes_of(t) for t in host_out], in_flight)
    for p in pools.values():
        p.shutdown()

    # ---- copy-only ceiling at this N: the same frames up and down on 8 streams, no kernels
    dbuf = [torch.empty(FRAME_BYTES, dtype=torch.uint8, device=dev) for _ in range(ne)]
    cstreams = [torch.cuda.Stream(device=dev) for _ in range(8)]

    def copy_step():
        for i in range(ne):
            with torch.cuda.stream(cstreams[i % 8]):
                dbuf[i].copy_(host_in[i], non_blocking=True)
                host_out[i].copy_(dbuf[i], non_blocking=True)
        torch.cuda.synchronize()
    ceiling = world * ne / timed_host(copy_step, args.steps, 2)
    torch.cuda.set_stream(tstream)

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cfps, cms, cores, cn = cpu_arm(8, 1)
        cpu = {"value": cfps, "unit": "frames/s", "cores": cores, "kind": "port",
               "sample": f"{cn} frames per step, 8 timed steps after 1 warm-up step, one frame per host thread ({cores} threads); " + CPU_NOTE}

    if rank == 0:
        line = {
            "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u16", "data": "synthetic",
            "config": CONFIG,
            "batch": {"frames_per_step_per_gpu": n, "bytes_per_step_per_gpu": 2 * n * FRAME_BYTES, "host_cores_per_rank": len(my_cores) if my_cores else None},
            "clocks": clocks,
            "e2e": {"value": e2e_pinned, "unit": "frames/s", "h2d_bytes_per_step": ne * FRAME_BYTES, "d2h_bytes_per_step": ne * FRAME_BYTES,
                    "frames_per_step_per_gpu": ne, "in_flight": in_flight,
                    "api": "vszip_boxblur_get_frame; value = frames in pinned host memory (the bench contract's definition of e2e), one DMA per direction",
                    "pageable": e2e_staged, "pageable_in_flight": in_flight_staged,
                    "pageable_note": "the same call on PAGEABLE planes that come back step after step, the way VapourSynth's frame pool hands them "
                                     "over: the library's default path (CPU copies through pinned staging buffers, both directions) - what a .vpy script gets",
                    "pageable_registered": e2e_registered, "registered_bytes": registered,
                    "pageable_registered_note": "opt-in host pin cache (vszip_cuda_host_register_limit): buffers that come back are page-locked in place",
                    "pcie_ceiling_fps": ceiling,
                    "pcie_ceiling_note": "copy-only probe in this run at this N: the same frames up and down on 8 streams per GPU, no kernels"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "algorithmic_bytes": ALGO_BYTES * n, "peak_source": peak_src,
                         "note": "algorithmic bytes = 12,441,600 B per frame (read once + write once) x frames per launch / launch duration"},
            "path": {"h_kernel_ms": ms_h, "v_kernel_ms": ms_v, "step_ms": ms_step, "algorithmic_GBps": path_gbs, "frac_of_peak": path_gbs / peak},
            "configs": configs,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def other_configs(vz, lib, torch, np, timed, timed_host, stream, world, peak, steps, headline, headline_gbs, my_cores):
    """BASELINE.json configs 1..5 at this N (every rank runs the same batch on its own GPU; fps is the whole job's)."""
    out = {}

    def entry(name, fmt, w, h, frames, algo_bytes_per_frame, ms, **more):
        f = world * frames / (ms * 1e-3)
        gbs = algo_bytes_per_frame * f / world / 1e9
        e = {"config": name, "format": fmt, "size": f"{w}x{h}", "frames_per_launch_per_gpu": frames, "fps": f, "us_per_frame_per_gpu": ms * 1e3 / frames,
             "algorithmic_bytes_per_frame": algo_bytes_per_frame, "GBps_per_gpu": gbs, "frac_of_hbm_peak": gbs / peak}
        e.update(more)
        return e

    def pixel(name, fmt, w, h, frames, make):
        a, b = vz.DeviceClip(fmt, w, h, frames), vz.DeviceClip(fmt, w, h, frames)
        a.fill_noise(1234)
        f = make(a)
        ms = timed(lambda: f.run_device(a, b, first=0, count=frames, stream=stream), steps, 3)
        e = entry(name, fmt, w, h, frames, 2 * a.frame_bytes, ms)
        a.free(); b.free()
        return e

    out["c1"] = pixel("configs[0]: BoxBlur 13/1/13/1 (comptime path, one read + one write)", "YUV420P16", 1920, 1080, 256,
                      lambda s: vz.BoxBlurFilter(s.info(), hradius=13, hpasses=1, vradius=13, vpasses=1))
    out["c2"] = {"config": "configs[1]: BoxBlur 13/5/13/5 [headline, see value/roofline/path]", "format": "YUV420P16", "size": "1920x1080",
                 "frames_per_launch_per_gpu": headline["frames"], "fps": headline["fps"], "us_per_frame_per_gpu": headline["ms_per_frame_batch"] * 1e3 / headline["frames"],
                 "algorithmic_bytes_per_frame": ALGO_BYTES, "GBps_per_gpu": headline_gbs, "frac_of_hbm_peak": headline_gbs / peak}
    out["c3"] = pixel("configs[2]: Bilateral sigmaS=2 sigmaR=2 planes=[0,1,2]", "YUV420P16", 1920, 1080, 128,
                      lambda s: vz.BilateralFilter(s.info(), sigmaS=2, sigmaR=2, planes=[0, 1, 2]))
    # the kernel is compute-bound, so the HBM fraction says little: the same measurement against the SM roofs that bind it
    # (sigmaS = 2 -> pattern (2,2): 16 taps per pixel = 16 MUFU.EX2 + 1 MUFU.RCP; 156 issued warp-instructions per pixel from the ncu
    # capture in profiles/ncu_bilateral_r02.md; per SM and clock: 16 MUFU lanes, 4 issue slots; DESIGN.md 4.3)
    props = torch.cuda.get_device_properties(torch.cuda.current_device())
    clock_hz = float(props.clock_rate) * 1e3 if getattr(props, "clock_rate", 0) else 1.965e9
    px_per_s = out["c3"]["fps"] / world * (1920 * 1080 * 1.5)
    sms = props.multi_processor_count
    out["c3"]["roofs"] = {"mufu_frac": px_per_s * 17 / (sms * 16 * clock_hz), "issue_frac": px_per_s * 156 / 32 / (sms * 4 * clock_hz),
                          "sm_clock_hz": clock_hz,
                          "note": "fractions of per-SM peaks at the SM's maximum clock: MUFU 16 lanes/clk, issue 4 warp-instructions/clk"}
    # configs[3]: PlaneMinMax + PlaneAverage with minthr/maxthr/exclude on 4K GRAYS and GRAY16; both results per frame
    c4 = {}
    for fmt, excl in (("GRAY16", [0, 32768]), ("GRAYS", [0, 1])):
        frames = 64
        a = vz.DeviceClip(fmt, 3840, 2160, frames)
        a.fill_noise(1234)
        mmf = vz.PlaneMinMaxFilter(a.info(), minthr=0.1, maxthr=0.1)
        avf = vz.PlaneAverageFilter(a.info(), exclude=excl)
        ms_mm = timed(lambda: vz._check(lib.vszip_planeminmax_device(mmf.handle, a.handle, None, 0, frames, None, stream)), steps, 3)
        ms_av = timed(lambda: vz._check(lib.vszip_planeaverage_device(avf.handle, a.handle, None, 0, frames, None, stream)), steps, 3)
        _, fused = vz.plane_stats_device(mmf, avf, a, count=frames, stream=stream, fetch=False)
        ms_both = timed(lambda: vz.plane_stats_device(mmf, avf, a, count=frames, stream=stream, fetch=False), steps, 3)
        fb = a.frame_bytes
        c4[fmt] = {"PlaneMinMax(minthr=.1,maxthr=.1)": entry("PlaneMinMax thr", fmt, 3840, 2160, frames, fb, ms_mm),
                   f"PlaneAverage(exclude={excl})": entry("PlaneAverage", fmt, 3840, 2160, frames, fb, ms_av),
                   "both (vszip_planestats_device)": entry("PlaneMinMax + PlaneAverage, one call", fmt, 3840, 2160, frames, fb, ms_both, one_read=bool(fused))}
        a.free()
    out["c4"] = {"config": "configs[3]: PlaneMinMax + PlaneAverage with minthr/maxthr/exclude on 3840x2160 GRAYS and GRAY16", **c4}

    # configs[4]: BoxBlur -> Bilateral -> PlaneMinMax on 3840x2160 YUV444PS, frame-parallel
    fmt, w, h, frames = "YUV444PS", 3840, 2160, 16
    a, b, c = (vz.DeviceClip(fmt, w, h, frames) for _ in range(3))
    a.fill_noise(1234)
    blur = vz.BoxBlurFilter(a.info(), hradius=13, hpasses=1, vradius=13, vpasses=1)
    bil = vz.BilateralFilter(a.info(), sigmaS=2, sigmaR=2)
    mm = vz.PlaneMinMaxFilter(a.info(), minthr=0.1, maxthr=0.1, planes=[0])
    ms_blur = timed(lambda: blur.run_device(a, b, count=frames, stream=stream), steps, 2)
    ms_bil = timed(lambda: bil.run_device(b, c, count=frames, stream=stream), steps, 2)
    ms_mm = timed(lambda: vz._check(lib.vszip_planeminmax_device(mm.handle, c.handle, None, 0, frames, None, stream)), steps, 2)

    def chain_dev():
        blur.run_device(a, b, count=frames, stream=stream)
        bil.run_device(b, c, count=frames, stream=stream)
        vz._check(lib.vszip_planeminmax_device(mm.handle, c.handle, None, 0, frames, None, stream))
    ms_chain = timed(chain_dev, steps, 2)
    fb = a.frame_bytes
    c5 = {"config": "configs[4]: BoxBlur(13,1,13,1) -> Bilateral(2,2) -> PlaneMinMax(.1,.1,planes=[0]) on 3840x2160 YUV444PS (bounded sample of the 5000-frame clip)",
          "BoxBlur": entry("BoxBlur 13/1/13/1 f32 (comptime float path)", fmt, w, h, frames, 2 * fb, ms_blur),
          "Bilateral": entry("Bilateral 2/2 f32", fmt, w, h, frames, 2 * fb, ms_bil),
          "PlaneMinMax": entry("PlaneMinMax thr plane 0", fmt, w, h, frames, fb // 3, ms_mm),
          "chain_device_resident": entry("three *_device calls on resident frames", fmt, w, h, frames, 4 * fb + fb // 3, ms_chain)}
    for d in (a, b, c):
        d.free()
    # end to end through the frame API: one fused vszip_chain_get_frame per frame (1 upload + 1 download), pinned frames
    ne = 8
    handles = (C.c_void_p * 3)(blur.handle, bil.handle, mm.handle)
    chain = lib.vszip_chain_create(handles, 3)
    if not chain:
        raise RuntimeError(vz._last_error())
    keep = []

    def pinned_frame(seed):
        t = torch.empty(3 * w * h * 4, dtype=torch.uint8).pin_memory()
        arr = t.numpy().view(np.float32).reshape(3, h, w)
        if seed is not None:
            r = np.random.default_rng(seed)
            arr[0] = r.random((h, w), dtype=np.float32)
            arr[1:] = r.random((2, h, w), dtype=np.float32) - np.float32(0.5)
        keep.append(t)
        return [arr[0], arr[1], arr[2]]
    fin = [vz._cframe(pinned_frame(i)) for i in range(ne)]
    fout = [vz._cframe(pinned_frame(None)) for _ in range(ne)]

    def one(i):
        o = vz._MinMaxProps()
        outs = (C.c_void_p * 3)(None, None, C.cast(C.pointer(o), C.c_void_p))
        if lib.vszip_chain_get_frame(chain, i, C.byref(fin[i]), C.byref(fout[i]), outs):
            raise RuntimeError(vz._last_error())
    threads = max(2, min(4, len(my_cores) if my_cores else 4))
    with ThreadPoolExecutor(threads) as ex:
        s = timed_host(lambda: list(ex.map(one, range(ne))), steps, 2)
    c5["e2e_fused_chain"] = {"fps": world * ne / s, "api": "vszip_chain_get_frame on pinned frames", "in_flight": threads,
                             "h2d_bytes_per_frame": 3 * w * h * 4, "d2h_bytes_per_frame": 3 * w * h * 4, "frames_per_step_per_gpu": ne}
    lib.vszip_chain_free(chain)
    del keep
    out["c5"] = c5
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=int(os.environ.get("WORLD_SIZE", "1")))
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config legs (configs c1..c5)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the headline's last-step output to DIR/*.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the CUDA arm's output; the reference arm runs on other inputs")
    # The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner there) must not add to it:
    # point fd 1 at stderr for the whole run and hand the real stdout to the two print(json.dumps(..)) calls only.
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_ours(args)
    finally:
        real_stdout.flush()


if __name__ == "__main__":
    main()
