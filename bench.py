#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: 4K YUY2 encode+decode fps per B200, wavelet HBM GB/s vs roofline.

A "step" = one pass of the hot path (forward 3-level 2-6 wavelet + quantise, then dequantise + inverse
3-level wavelet) over one batch of synthetic 3840x2160 YUY2 frames.

  value   : whole-job throughput, frames (encode+decode pairs) per second, inputs resident in HBM,
            kernels only, CUDA events on the launching stream, max over ranks.
  e2e     : the same metric through the C ABI with HOST buffers: the asynchronous in-order frame pool
            (cfb_pool_submit_forward_sparse / _inverse_sparse + cfb_pool_wait).  Every frame is copied H2D from
            pinned host memory, its coefficients come back D2H (lossless sparse format), go H2D again for the
            decode and the decoded frame is copied D2H; all copies are inside the timed region.  The dense
            int16 format (cfb_pool_submit_forward / _inverse) is reported next to it.
  roofline: the dominant kernel (level-1 forward, k_fwd_422) timed alone, live, with CUDA events.
  cpu_baseline / --impl reference: the reference's own calls for this path (oracle/_ref, the unmodified
            reference compiled in place) on the box's host cores.

Multi-GPU: frames are independent (GOP 1) -> each rank owns its own frames, no data-path collective;
torch.distributed (NCCL) is used only for the barrier and the max-over-ranks of the timing.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

QUALITY = 4                                       # FILMSCAN1
# --config: the BASELINE.json configurations that are GPU bench lines.  Default = configs[2], the one the metric is quoted on.
CONFIGS = {
    "yuv422": dict(width=3840, height=2160, fmt="YUYV", batch=16, decode=True, metric="4K YUY2 encode+decode fps",
                   workload="TestCFHD -E/-D 3840x2160 YUY2 4:2:2 (BASELINE.json configs[2]), FILMSCAN1, GOP 1, progressive"),
    "rgb444": dict(width=3840, height=2160, fmt="RG48", batch=8, decode=False, inverse_levels=True, metric="4K RGB 4:4:4 12-bit encode fps",
                   workload="3840x2160 RGB 4:4:4 12-bit (3-channel, RG48 source) encode (BASELINE.json configs[3]), FILMSCAN1, GOP 1"),
    "bayer8k": dict(width=7680, height=4320, fmt="BYR4", batch=4, decode=False, metric="8K Bayer RAW encode fps",
                    workload="7680x4320 16-bit Bayer RAW (BYR4, curve applied) encode (BASELINE.json configs[4]), FILMSCAN1, GOP 1"),
}
CFG = CONFIGS["yuv422"]
WIDTH, HEIGHT, METRIC, WORKLOAD = CFG["width"], CFG["height"], CFG["metric"], CFG["workload"]


def select_config(name):
    global CFG, WIDTH, HEIGHT, METRIC, WORKLOAD
    CFG = CONFIGS[name]
    WIDTH, HEIGHT, METRIC, WORKLOAD = CFG["width"], CFG["height"], CFG["metric"], CFG["workload"]


def ncu_traffic_per_launch(kernel_summary):
    """DRAM bytes (read + write) of one launch of the dominant kernel from the committed `ncu --set full` capture
    (profiles/<round>_prof_*_summary.csv, taken with the same 16-frame batch); None if the summary is absent."""
    path = os.path.join(ROOT, "profiles", kernel_summary)
    try:
        vals = {}
        for line in open(path):
            k, unit, v = line.rstrip("\n").split(",")[:3]
            if k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                vals[k] = float(v) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[unit]
        return int(vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"])
    except Exception:
        return None


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------
class Dist:
    """torch.distributed plumbing of the benchmark: barrier + max-over-ranks of the device timing.  The data path
    never uses it (frames are independent: SURVEY 8e).  backend "nccl" on GPUs, "gloo" in the CPU tests."""

    def __init__(self, world, backend="nccl", local_rank=0):
        self.world, self.backend, self.local_rank = world, backend, local_rank
        self.dist = None
        if world > 1:
            import torch
            import torch.distributed as dist
            kw = {"device_id": torch.device("cuda", local_rank)} if backend == "nccl" else {}
            dist.init_process_group(backend, **kw)
            self.dist = dist

    def barrier(self):
        if self.dist:
            self.dist.barrier()

    def max(self, x):
        if not self.dist:
            return float(x)
        import torch
        t = torch.tensor([float(x)], device="cuda" if self.backend == "nccl" else "cpu")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist:
            self.dist.destroy_process_group()


def aggregate_fps(world, frames_per_rank, max_seconds):
    """Whole-job throughput: every rank processed frames_per_rank frames within the slowest rank's time."""
    return world * frames_per_rank / max_seconds


def shard_seed(rank):
    """Each rank/GPU encodes its own frames (weak scaling): distinct buffers per rank."""
    return 1000 * rank


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
                "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [l.strip().split(", ") for l in open(self.path) if l.strip()]
            sm = sorted(int(r[0]) for r in rows if r[0].isdigit())
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = int(rows[0][1])
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for k, n in enumerate(names):
                if any(len(r) > 2 + k and r[2 + k].strip().lower() == "active" for r in rows):
                    out["reasons"].append(n)
            out["samples"] = len(sm)
        except Exception:
            pass
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        return out


# ------------------------------------------------------------------------------------------------
DATA_NOTE = ("synthetic (deterministic procedural frames: smooth illumination + 1/f oriented sinusoids over eight octaves + "
             "hard-edged shapes + faint grain; about 30 % more non-zero coefficients per 4K frame at FILMSCAN1 than "
             "TestCFHD's Qbist frames, i.e. conservative for the sparse transfer path)")


def procedural_frame(width, height, variant=0):
    """Deterministic 8-bit 4:2:2 test frame: smooth illumination, a 1/f sum of oriented sinusoids over eight octaves,
    hard-edged discs and bars, and a faint fixed grain.  Scale-aware (features are defined in pixels of a 1920-wide frame
    and grow with the width) so that the coefficient statistics per pixel are those of a natural image at any size."""
    rng = np.random.default_rng(1000 + variant)
    s = width / 1920.0
    yy, xx = np.meshgrid(np.arange(height, dtype=np.float32), np.arange(width, dtype=np.float32), indexing="ij")
    u, v = xx / width, yy / height
    Y = 0.45 + 0.25 * np.sin(2.1 * u + 0.7 * variant) * np.cos(1.7 * v) + 0.10 * u - 0.05 * v
    Cb = 0.08 * np.sin(3.0 * u + 1.3) + 0.05 * v
    Cr = 0.08 * np.cos(2.3 * v + 0.4) - 0.04 * u
    for octave in range(8):
        f = (2.0 ** octave) * 2.0 * np.pi / (1920.0 * s) * 1.5            # radians per pixel
        amp = 0.12 / (1.6 ** octave)
        for _ in range(2):
            th, ph = rng.uniform(0, np.pi), rng.uniform(0, 2 * np.pi)
            wave = np.sin(f * (np.cos(th) * xx + np.sin(th) * yy) + ph)
            Y += amp * wave
            if octave < 4:
                Cb += 0.35 * amp * np.sin(f * (np.cos(th + 1.0) * xx + np.sin(th + 1.0) * yy) + ph)
                Cr += 0.35 * amp * np.cos(f * (np.cos(th - 1.0) * xx + np.sin(th - 1.0) * yy) + ph)
    for _ in range(14):                                                    # hard edges: discs and bars
        cx, cy, r = rng.uniform(0, width), rng.uniform(0, height), rng.uniform(20, 160) * s
        dy, dcb = rng.uniform(-0.25, 0.25), rng.uniform(-0.08, 0.08)
        if rng.random() < 0.5:
            m = (xx - cx) ** 2 + (yy - cy) ** 2 < r * r
        else:
            m = (np.abs(xx - cx) < r) & (np.abs(yy - cy) < 0.35 * r)
        Y = np.where(m, Y + dy, Y); Cb = np.where(m, Cb + dcb, Cb); Cr = np.where(m, Cr - dcb, Cr)
    grain = ((xx.astype(np.int64) * 73856093) ^ (yy.astype(np.int64) * 19349663) ^ (variant * 83492791)) & 7
    Y = Y + (grain.astype(np.float32) - 3.5) * (1.0 / 255.0) * 0.6
    out = np.zeros((height, width * 2), np.uint8)
    out[:, 0::2] = np.clip(16 + 219 * np.clip(Y, 0, 1) + 0.5, 0, 255).astype(np.uint8)
    out[:, 1::4] = np.clip(128 + 224 * 0.5 * (Cb[:, 0::2] + Cb[:, 1::2]) + 0.5, 16, 240).astype(np.uint8)
    out[:, 3::4] = np.clip(128 + 224 * 0.5 * (Cr[:, 0::2] + Cr[:, 1::2]) + 0.5, 16, 240).astype(np.uint8)
    return out


def psnr(a, b):
    mse = np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2)
    return 99.0 if mse == 0 else 10 * np.log10(255.0 ** 2 / mse)


_BASE_FRAMES = {}


def synthetic_frames(n, width, height, seed=0):
    """n frame buffers for the benchmark, generated here (no test infrastructure, no reference code on the product arm).
    Two distinct base frames; the n buffers are distinct memory (cyclic row shifts of the bases) so that every step
    streams more than the L2 of fresh data.  TestCFHD -E itself re-submits one Qbist frame 500x (TestCFHD.cpp:957)."""
    key = (width, height)
    if key not in _BASE_FRAMES:
        _BASE_FRAMES[key] = [procedural_frame(width, height, v) for v in range(2)]
    bases = _BASE_FRAMES[key]
    return [np.ascontiguousarray(np.roll(bases[i % len(bases)], (16 * i + 6 * seed + 2 * (seed // 1000)) % height, axis=0)) for i in range(n)]


def procedural_rgb48(width, height, variant=0):
    """16-bit packed RGB (RG48) rendition of procedural_frame: BT.709 conversion of its Y'CbCr planes to full-range RGB,
    12 significant bits plus a deterministic low-order texture (height x 3*width uint16)."""
    f = procedural_frame(width, height, variant).astype(np.float32)
    y = (f[:, 0::2] - 16.0) / 219.0
    cb = np.repeat((f[:, 1::4] - 128.0) / 224.0, 2, axis=1)
    cr = np.repeat((f[:, 3::4] - 128.0) / 224.0, 2, axis=1)
    r, g, b = y + 1.5748 * cr, y - 0.1873 * cb - 0.4681 * cr, y + 1.8556 * cb
    yy, xx = np.meshgrid(np.arange(height, dtype=np.int64), np.arange(width, dtype=np.int64), indexing="ij")
    tex = (((xx * 2654435761) ^ (yy * 40503)) & 0xFF).astype(np.float32)
    out = np.zeros((height, width * 3), np.uint16)
    for i, c in enumerate((r, g, b)):
        out[:, i::3] = (np.clip(c, 0.0, 1.0) * 65280.0 + tex).astype(np.uint16)
    return out


def procedural_bayer(width, height, variant=0):
    """16-bit Bayer mosaic (RED_GRN phase: r g / g b), curve already applied: the RG48 frame at half the size, each
    pixel seen through the colour filter array, pixel-doubled with a small position-dependent offset."""
    rgb = procedural_rgb48(width // 2, height // 2, variant)
    r = np.repeat(np.repeat(rgb[:, 0::3], 2, axis=0), 2, axis=1).astype(np.int32)
    g = np.repeat(np.repeat(rgb[:, 1::3], 2, axis=0), 2, axis=1).astype(np.int32)
    b = np.repeat(np.repeat(rgb[:, 2::3], 2, axis=0), 2, axis=1).astype(np.int32)
    yy, xx = np.meshgrid(np.arange(height, dtype=np.int64), np.arange(width, dtype=np.int64), indexing="ij")
    off = (((xx * 97) ^ (yy * 57)) & 0x3F).astype(np.int32) * 16
    m = np.empty((height, width), np.int32)
    m[0::2, 0::2] = r[0::2, 0::2]; m[0::2, 1::2] = g[0::2, 1::2]
    m[1::2, 0::2] = g[1::2, 0::2]; m[1::2, 1::2] = b[1::2, 1::2]
    return np.clip(m + off, 0, 65535).astype(np.uint16)


def config_frames(n, seed=0):
    """n distinct input buffers of the selected config (uint8 views, rows x pitch bytes)."""
    fmt = CFG["fmt"]
    if fmt == "YUYV":
        return synthetic_frames(n, WIDTH, HEIGHT, seed)
    key = (WIDTH, HEIGHT, fmt)
    if key not in _BASE_FRAMES:
        gen = procedural_rgb48 if fmt == "RG48" else procedural_bayer
        _BASE_FRAMES[key] = [gen(WIDTH, HEIGHT, v) for v in range(2)]
    bases = _BASE_FRAMES[key]
    step = 16 if fmt == "RG48" else 32                  # Bayer: keep the colour-filter phase (even shifts)
    return [np.ascontiguousarray(np.roll(bases[i % 2], (step * i + 6 * seed + 2 * (seed // 1000)) % HEIGHT, axis=0)).view(np.uint8)
            for i in range(n)]


def cpu_reference_run(width, height, quality, threads, iters):
    """Times the reference's own transform calls (oracle/_ref) on `threads` host threads, `iters` frames each.
    Returns (frames_per_second, kind, sample_description)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))         # the checker (oracle/, tests/) is used by this leg only
    import oracle_lib as ol
    import parity_util as pu
    if CFG["fmt"] != "YUYV":
        return cpu_reference_run_planar(ol, width, height, quality, threads, iters)
    frame = synthetic_frames(1, width, height)[0]
    if ol.ref_available():
        ref = ol.load_ref()
        results = [None] * threads

        def work(t):
            f, i = C.c_double(), C.c_double()
            rc = ref.ref_time_transform_422(frame.ctypes.data_as(C.c_void_p), width, height, width * 2, quality,
                                            iters, 1, C.byref(f), C.byref(i), None)
            results[t] = (rc, f.value, i.value)

        t0 = time.perf_counter()
        ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
        [t.start() for t in ths]
        [t.join() for t in ths]
        wall = time.perf_counter() - t0
        assert all(r and r[0] == 0 for r in results), "reference timing probe failed"
        # the probe's setup (one full encode + decode per thread) is outside its own timed loops:
        busy = max(r[1] + r[2] for r in results)
        fps = threads * iters / busy
        desc = (f"{threads} threads x {iters} frames, each: TransformForwardSpatialYUV + ComputeGroupTransformQuant, then "
                f"ReconstructWaveletBand x2/channel + ReconstructSampleFrameToBuffer (8-bit YUYV); unmodified reference, "
                f"gcc -O2 -msse2; wall {wall:.1f}s incl. setup")
        return fps, "reference", desc
    # port: the scalar C restatement (single thread)
    orc = ol.oracle()
    pkg = importlib.import_module("cineform-sdk_b200")
    q = pkg.quant_for_quality(pkg.FrameDesc(width, height, pkg.PIXEL_YUYV), quality)
    t0 = time.perf_counter()
    bands = pu.oracle_forward_422(orc, frame, q, 0)
    pu.inverse_pyramid(orc, bands, q.table(3), tuple(q.prescale))
    dt = time.perf_counter() - t0
    return 1.0 / dt, "port", "1 frame forward+inverse with oracle/liboracle.so (scalar C restatement), 1 thread"


def cpu_reference_run_planar(ol, width, height, quality, threads, iters):
    """configs 4 / 5: the reference's forward path for a planar source (conversion + level 1 per plane + levels 2, 3) on
    `threads` host threads (oracle/ref_probe.cpp ref_time_forward_planar)."""
    if not ol.ref_available():
        raise SystemExit("bench.py --impl reference --config %s needs oracle/_ref (the reference compiled in place)" % CFG["fmt"])
    ref = ol.load_ref()
    frame = config_frames(1)[0]
    if CFG["fmt"] == "BYR4":
        w, h, pitch, cf, nch = width // 2, height // 2, width * 4, 104, 4       # plane dimensions, doubled pitch (SampleEncoder.cpp:494)
        ref.ref_set_bayer_format(0)
    else:
        w, h, pitch, cf, nch = width, height, width * 6, 120, 3
    results = [None] * threads

    def work(t):
        f = C.c_double()
        rc = ref.ref_time_forward_planar(frame.ctypes.data_as(C.c_void_p), w, h, pitch, cf, nch, quality, iters, C.byref(f))
        results[t] = (rc, f.value)

    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    wall = time.perf_counter() - t0
    if CFG["fmt"] == "BYR4":
        ref.ref_set_bayer_format(-1)
    assert all(r and r[0] == 0 for r in results), "reference timing probe failed"
    fps = threads * iters / max(r[1] for r in results)
    conv = "ConvertBYR4ToFrame16s" if CFG["fmt"] == "BYR4" else "ConvertRGB48ToFrame16s"
    desc = (f"{threads} threads x {iters} frames, each: {conv} + TransformForwardSpatial per plane + ComputeGroupTransformQuant "
            f"(encode only); unmodified reference, gcc -O2 -msse2; wall {wall:.1f}s incl. setup")
    return fps, "reference", desc


# ------------------------------------------------------------------------------------------------
def usable_cpus():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota (containers), not just nproc."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return max(1, n)


def reference_best(iters):
    """The reference's best configuration on this box: its transform path is timed with several host-thread counts
    (every thread owns an ENCODER + DECODER, like the reference's own EncoderPool workers) and the fastest result is
    reported.  More threads than the cgroup CPU quota only thrash, so the candidates stop at the usable core count.
    `iters` scales the sample (frames per thread at the largest thread count)."""
    ncpu = usable_cpus()
    best = None
    for t in sorted({max(1, ncpu // 4), max(1, ncpu // 2), ncpu}):
        per_thread = max(2, iters * ncpu // t)
        fps, kind, desc = cpu_reference_run(WIDTH, HEIGHT, QUALITY, t, per_thread)
        if best is None or fps > best[0]:
            best = (fps, kind, desc, t)
    fps, kind, desc, t = best
    return fps, kind, desc + f"; best of thread counts up to the {ncpu} usable cores (os.cpu_count() = {os.cpu_count()})", t


def arm_config(args):
    """The `config` object is identical on both arms (ours / --impl reference): same workload, same stage."""
    return {"workload": WORKLOAD, "name": args.config,
            "stage": "wavelet + quantisation transform path only (entropy coding stays on the host and is excluded on both arms); "
                     + ("encode + decode of every frame" if CFG["decode"] else "encode of every frame")}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores.
    Step 0 picks the fastest host-thread count (reference_best); every later step re-times that configuration on a
    sample sized so that the whole --steps/--warmup run stays inside --ref-budget-s of wall clock."""
    if rank != 0:
        return
    t_start = time.perf_counter()
    total = args.warmup + args.steps
    fps0, kind, desc, threads = reference_best(max(1, args.ref_iters))
    results = [(fps0, desc)] if args.warmup == 0 else []
    per_frame_s = threads / fps0                 # one thread's time for one frame (forward + inverse)
    setup_s = 1.5                                # probe set-up per call (one real encode + decode per thread), measured below
    for s in range(1, total):
        remaining = args.ref_budget_s - (time.perf_counter() - t_start)
        slot = max(0.0, remaining) / (total - s)
        iters = int(max(1, min(args.ref_iters * 4, (slot - setup_s) / per_frame_s)))
        t0 = time.perf_counter()
        fps, kind, d = cpu_reference_run(WIDTH, HEIGHT, QUALITY, threads, iters)
        setup_s = max(0.2, (time.perf_counter() - t0) - iters * threads / fps)
        if s >= args.warmup:
            results.append((fps, d))
    fps, desc = max(results, key=lambda r: r[0])
    frames = int(desc.split(" threads x ")[1].split(" frames")[0]) * threads
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "fps", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * frames / fps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int16", "data": DATA_NOTE,
        "config": arm_config(args),
        "config_details": {"frames_per_step": frames,
                           "sampling": f"best of {len(results)} timed steps; thread count chosen in step 0 from "
                                       f"{{1/4, 1/2, 1}} x usable cores; wall {time.perf_counter() - t_start:.0f}s "
                                       f"(budget {args.ref_budget_s}s)"},
        "cpu_baseline": {"value": fps, "unit": "fps", "cores": threads, "kind": kind, "sample": desc},
        "e2e": {"value": fps, "unit": "fps", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
def copy_ceiling(torch, up_bytes, down_bytes, seconds=0.6):
    """What the copy engines sustain for the e2e copy pattern of this config on THIS box: per unit of work the given
    byte lists are copied H2D / D2H between pinned host buffers and device memory on two streams, nothing else runs.
    Every rank measures at the same time, so at N > 1 the figure includes the host-side contention (NUMA node, root
    complex) that bounds the N-GPU e2e number.  Returns units per second."""
    ring = 24
    hu = [[torch.empty(b, dtype=torch.uint8).pin_memory() for b in up_bytes] for _ in range(ring)]
    hd = [[torch.empty(b, dtype=torch.uint8).pin_memory() for b in down_bytes] for _ in range(ring)]
    du = [[torch.empty(b, dtype=torch.uint8, device="cuda") for b in up_bytes] for _ in range(4)]
    dd = [[torch.empty(b, dtype=torch.uint8, device="cuda") for b in down_bytes] for _ in range(4)]
    s_up, s_dn = torch.cuda.Stream(), torch.cuda.Stream()

    def run(n):
        torch.cuda.synchronize(); t = time.perf_counter()
        for i in range(n):
            with torch.cuda.stream(s_up):
                for dst, src in zip(du[i % 4], hu[i % ring]):
                    dst.copy_(src, non_blocking=True)
            with torch.cuda.stream(s_dn):
                for dst, src in zip(hd[i % ring], dd[i % 4]):
                    dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        return time.perf_counter() - t

    run(8)
    probe = run(32)
    n = max(32, int(32 * seconds / probe))
    return n / run(n)


def dump_outputs(out_dir, outputs, budget_bytes=60 << 20):
    """Writes what the timed path returned as out_dir/<name>.npy (float32, exact for these integer types).
    outputs: {name: (device uint8 buffers, numpy dtype, elements per buffer)}; the buffers are concatenated in order.
    An output larger than its share of the budget is written as a fixed sample: element indices drawn with a seeded
    generator and sorted, so two runs with the same arguments sample the same elements."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = budget_bytes // 4 // len(outputs)
    for name, (bufs, dtype, n) in outputs.items():
        dtype = np.dtype(dtype)
        total = len(bufs) * n
        idx = None if total <= cap else np.unique(np.random.default_rng(0).integers(0, total, cap))
        parts = []
        for i, buf in enumerate(bufs):
            v = buf[:n * dtype.itemsize].view(torch.uint8 if dtype.itemsize == 1 else torch.int16)
            if idx is not None:
                sel = idx[(idx >= i * n) & (idx < (i + 1) * n)] - i * n
                v = v[torch.from_numpy(sel).to(v.device)]
            parts.append(v.cpu().numpy().view(dtype))
        np.save(os.path.join(out_dir, name + ".npy"), np.concatenate(parts).astype(np.float32))


def run_ours(args, rank, world, local_rank):
    import torch
    pkg = importlib.import_module("cineform-sdk_b200")        # raises if libcfhd_b200.so is missing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the transform path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    D = Dist(world, "nccl", local_rank)
    barrier = D.barrier

    # one process per GPU, placed on the GPU's own NUMA node (as `numactl --cpunodebind` would): pinned buffers
    # allocated below and the pool's threads are then local to the PCIe root of this rank's GPU.  The original mask
    # is restored before the CPU baseline so that the reference arm keeps every host core.
    full_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_node = pkg.device_numa_node(local_rank)
    if not args.no_numa_bind:
        pkg.bind_thread_to_device(local_rank)

    B = args.batch or CFG["batch"]
    fmt = getattr(pkg, "PIXEL_" + CFG["fmt"])
    decode = CFG["decode"]
    out_fmt = {"YUYV": pkg.PIXEL_YUYV, "RG48": pkg.PIXEL_RG48}.get(CFG["fmt"], pkg.PIXEL_PLANAR16)
    ctx = pkg.Context(local_rank)
    desc = pkg.FrameDesc(WIDTH, HEIGHT, fmt)
    quant = pkg.quant_for_quality(desc, QUALITY)
    codec = pkg.Codec(ctx, desc, B)
    lay = codec.layout
    stream = torch.cuda.ExternalStream(ctx.stream)
    frames = config_frames(B, seed=shard_seed(rank))

    # ---- device-resident working set: B frames in, B pyramids, B frames out (>> 126 MB L2) ----
    with torch.cuda.stream(stream):
        d_in = [torch.from_numpy(f.reshape(-1)).cuda(non_blocking=False) for f in frames]
        d_pyr = [torch.zeros(lay.total_bytes, dtype=torch.uint8, device="cuda") for _ in range(B)]
        inv_levels = decode or CFG.get("inverse_levels", False)     # time the inverse kernels per level even when a step is encode-only
        d_out = [torch.zeros(lay.frame_bytes, dtype=torch.uint8, device="cuda") for _ in range(B)] if inv_levels else []
    ip, pp, op = [t.data_ptr() for t in d_in], [t.data_ptr() for t in d_pyr], [t.data_ptr() for t in d_out]
    ctx.synchronize()

    def fwd():
        codec.forward_device(ip, lay.frame_pitch, quant, pp)

    def inv():
        codec.inverse_device(pp, quant, out_fmt, op, lay.frame_pitch)

    def step_device():
        fwd()
        if decode:
            inv()

    def timed(fn, warmup, steps):
        for _ in range(warmup):
            fn()
        ctx.synchronize(); torch.cuda.synchronize(); barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        ctx.synchronize(); torch.cuda.synchronize(); barrier()
        return D.max(e0.elapsed_time(e1))

    # nvidia-smi clock / throttle sampling runs from here until the end of the e2e section, i.e. across every timed
    # region of this run (device-resident steps, per-kernel roofline timing, pooled e2e stream)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ctx.stats()["kernel_launches"]
    total_ms = timed(step_device, args.warmup, args.steps)
    launches_per_step = (ctx.stats()["kernel_launches"] - launches0) // (args.warmup + args.steps)
    launches = launches_per_step * args.steps
    ms_per_step = total_ms / args.steps
    value = aggregate_fps(world, B * args.steps, total_ms / 1000.0)
    if args.dump_outputs and rank == 0:
        # the last timed step's results, before the per-level timing below overwrites the buffers
        outputs = {"coefficients": (d_pyr, np.int16, lay.coded_bytes // 2)}
        if decode:
            out_dtype = {"YUYV": np.uint8, "RG48": np.uint16}.get(CFG["fmt"], np.int16)
            outputs["decoded"] = (d_out, out_dtype, lay.frame_bytes // np.dtype(out_dtype).itemsize)
        dump_outputs(args.dump_outputs, outputs)

    # ---- parity spot check of what was just timed (decoded frame vs input) ----
    roundtrip_psnr = None
    if inv_levels and not decode:
        inv(); ctx.synchronize()
    if CFG["fmt"] == "YUYV":
        with torch.cuda.stream(stream):
            back = d_out[0].cpu().numpy().reshape(HEIGHT, -1)
        roundtrip_psnr = psnr(back[:, 0::2], frames[0][:, 0::2])
    elif CFG["fmt"] == "RG48":
        with torch.cuda.stream(stream):
            back = d_out[0].cpu().numpy().view(np.uint16)
        a16, b16 = back.astype(np.float64)[:WIDTH * 3 * 64], frames[0].reshape(-1).view(np.uint16).astype(np.float64)[:WIDTH * 3 * 64]
        roundtrip_psnr = 10 * np.log10(65535.0 ** 2 / max(np.mean((a16 - b16) ** 2), 1e-9))

    # ---- roofline: every level of the pyramid timed alone ("HBM GB/s vs level"), the dominant kernel first ----
    P = sum(lay.band[c][0][0].width * lay.band[c][0][0].height * 4 for c in range(lay.num_channels))     # samples of all channels
    peak, peak_src = peaks()
    kname = {"YUYV": ("k_fwd_422_tma (TMA-staged packed 4:2:2 -> 12 bands, fused quant)", "k_inv_422"),
             "RG48": ("k_fwd_rg48 x3 (one launch per channel)", "k_inv_444_rg48"),
             "BYR4": ("k_fwd_byr4 (4 channels from the Bayer quads)", "-")}[CFG["fmt"]]
    levels = []
    reps = max(10, args.steps)
    for direction in ("forward", "inverse") if inv_levels else ("forward",):
        for lvl in (1, 2, 3):
            bit = 1 << (lvl - 1)
            if direction == "forward":
                codec.set_level_mask(bit, 0); fn = fwd
            else:
                codec.set_level_mask(0, bit); fn = inv
            ms = timed(fn, 3, reps) / reps
            algo = ((lay.frame_bytes + 2 * P) if lvl == 1 else (P // (4 ** (lvl - 2)) if lvl == 2 else P // 4)) * B
            gbs = algo / (ms * 1e-3) / 1e9
            levels.append({"direction": direction, "level": lvl, "kernel_ms": ms, "algorithmic_bytes_per_launch": int(algo),
                           "achieved": gbs, "frac": gbs / peak,
                           "kernel": (kname[0] if direction == "forward" else kname[1]) if lvl == 1 else
                                     ("k_fwd_plane" if direction == "forward" else "k_inv_plane") + ("<prescale 2>" if quant.prescale[lvl - 1] else "<0>")})
    codec.set_level_mask(7, 7)
    dom = levels[0]

    # ---- e2e through the C ABI with pinned host buffers: the asynchronous frame pool ----
    # Every frame is encoded (H2D packed frame, kernels, D2H coded coefficients) and -- configs that decode -- as soon as
    # its coefficients are back in host memory, decoded (H2D coefficients, kernels, D2H packed frame); encode and decode
    # jobs of different frames are in flight together so both PCIe directions stay busy.
    e2e = None
    if not args.no_e2e:
        sparse_ok = (CFG["fmt"] == "YUYV")             # the sparse inverse produces packed 4:2:2; other formats decode from dense bands
        ring = max(48, min(96, args.pool_inflight + 32)) if CFG["fmt"] == "YUYV" else 24
        pool = pkg.Pool([local_rank], desc, slots=args.pool_slots, batch=args.pool_batch,
                        queue_length=args.pool_inflight + 16)     # the bounded queue must never block this single submit/wait thread
        h_in = [pkg.pinned_empty((lay.frame_bytes // lay.frame_pitch, lay.frame_pitch)) for _ in range(ring)]
        h_cd = [pkg.pinned_empty(pkg.sparse_max_bytes(lay)) for _ in range(ring)]
        h_out = [pkg.pinned_empty((lay.frame_bytes // lay.frame_pitch, lay.frame_pitch)) for _ in range(ring)] if decode else []
        for i in range(ring):
            h_in[i][:] = frames[i % B].reshape(h_in[i].shape)

        def run_stream(total, sparse):
            sub_f = pool.submit_forward_sparse if sparse else pool.submit_forward
            sub_i = pool.submit_inverse_sparse if (sparse and sparse_ok) else pool.submit_inverse
            FWD, INV = 0, 1 << 30
            next_f, done = 0, 0
            inflight = 0
            while done < total:
                while next_f < total and inflight < args.pool_inflight and next_f - done < ring - 8:
                    sub_f(FWD | next_f, h_in[next_f % ring], quant, h_cd[next_f % ring])
                    next_f += 1; inflight += 1
                r = pool.wait(); inflight -= 1
                if (r & INV) or not decode:
                    done += 1
                else:
                    sub_i(INV | r, h_cd[r % ring], quant, out_fmt, h_out[r % ring])
                    inflight += 1

        def timed_stream(sparse, seconds):
            run_stream(2 * B, sparse)                   # warm-up (also teaches the pool the sparse payload size)
            t0 = time.perf_counter(); run_stream(4 * B, sparse); probe = time.perf_counter() - t0
            total = max(4 * B, int(4 * B * seconds / probe))
            barrier()
            before = pool.stats()
            t0 = time.perf_counter()
            run_stream(total, sparse)
            dt = D.max(time.perf_counter() - t0)
            after = pool.stats()
            if CFG["fmt"] == "YUYV":
                assert psnr(h_out[0][:, 0::2], h_in[0][:, 0::2]) > 40.0
            # bytes the copy engines really moved per frame (the speculative sparse download copies its size guess, not the exact size)
            moved = ((after["h2d_bytes"] - before["h2d_bytes"]) / total, (after["d2h_bytes"] - before["d2h_bytes"]) / total)
            return total, dt, moved

        sparse_fwd = sparse_ok or not decode            # encode-only configs can always use the sparse download
        n_dense, dt_dense, _ = timed_stream(False, min(1.0, args.e2e_seconds)) if sparse_fwd else (0, 1.0, None)
        nfr, dt_main, moved = timed_stream(sparse_fwd, args.e2e_seconds)
        coded_bytes = int(np.mean([pkg.sparse_bytes(h_cd[i]) for i in range(min(ring, B))])) if sparse_fwd else int(lay.coded_bytes)
        pool_stats = pool.stats()
        pool.close()
        del h_in, h_cd, h_out
        copied = int(moved[1] - (lay.frame_bytes if decode else 0)) if sparse_fwd else coded_bytes     # sparse D2H incl. the speculative margin
        up = [lay.frame_bytes] + ([coded_bytes] if decode else [])
        down = [copied] + ([lay.frame_bytes] if decode else [])
        barrier()
        ceiling = copy_ceiling(torch, up, down)
        ceiling_all = D.max(-ceiling)                   # the slowest rank bounds the job
        ceiling_fps = -ceiling_all * world
        e2e_value = aggregate_fps(world, nfr, dt_main)
        e2e = {"value": e2e_value, "unit": "fps",
               "h2d_bytes_per_step": int(B * moved[0]), "d2h_bytes_per_step": int(B * moved[1]),
               "bytes_source": "cfb_pool_stats deltas over the timed region (what the copy engines moved, incl. the margin of the speculative sparse download)",
               "api": f"cfb_pool_submit_forward{'_sparse' if sparse_fwd else ''}"
                      f"{('/inverse' + ('_sparse' if sparse_ok else '')) if decode else ''} + cfb_pool_wait (C ABI), pinned host buffers, "
                      f"{args.pool_slots} staging slots x batch {args.pool_batch} per GPU on three streams (upload / compute / download), "
                      f"{'encode and decode jobs interleaved' if decode else 'encode only'}{'' if args.no_numa_bind else f', rank bound to NUMA node {numa_node} of its GPU'}; "
                      f"coefficients cross PCIe as {'the lossless sparse format (two-level bitmaps + one byte per non-zero coefficient, escapes for |v| > 127)' if sparse_fwd else 'dense int16 bands'}, "
                      f"{coded_bytes} B/frame vs {lay.coded_bytes} dense",
               "frames": nfr, "seconds": dt_main, "per_gpu": e2e_value / world,
               "copy_ceiling": {"value": ceiling_fps, "unit": "fps", "frac": e2e_value / ceiling_fps,
                                "how": "the same H2D / D2H byte pattern per frame, copies only (two streams, pinned buffers, no kernels), "
                                       "measured by every rank at the same time right after the e2e run; min over ranks x ranks"},
               "limiter": "PCIe / host DMA: the copy engines are the bound (see copy_ceiling); SM time is "
                          f"{100.0 * (ms_per_step / 1e3 / B) * (e2e_value / world):.0f} % of the e2e wall time",
               "pool_kernel_launches": int(pool_stats["kernel_launches"])}
        if sparse_fwd:
            e2e["dense_format"] = {"value": aggregate_fps(world, n_dense, dt_dense), "unit": "fps",
                                   "h2d_bytes_per_step": int(B * (lay.frame_bytes + (lay.coded_bytes if decode else 0))),
                                   "d2h_bytes_per_step": int(B * (lay.coded_bytes + (lay.frame_bytes if decode else 0)))}

    clocks = sampler.stop() if rank == 0 else None
    if full_affinity is not None:
        os.sched_setaffinity(0, full_affinity)

    # ---- CPU baseline (rank 0, N == 1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fps, kind, descr, threads = reference_best(args.ref_iters)
        cpu = {"value": fps, "unit": "fps", "cores": threads, "kind": kind, "sample": descr}

    if rank == 0:
        traffic_csv = "r02_prof_fwd422_tma_summary.csv"
        line = {
            "metric": METRIC, "value": value, "unit": "fps", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int16", "data": DATA_NOTE if CFG["fmt"] == "YUYV" else DATA_NOTE + "; RG48 / Bayer frames derived from the same procedural image",
            "value_scope": "device-resident wavelet + quantisation kernels only (inputs in HBM; no PCIe, no entropy coding); the "
                           "host-to-host figure through the C ABI is `e2e`",
            "config": arm_config(args),
            "config_details": {"frames_per_step_per_gpu": B, "global_frames_per_step": B * world,
                       "parallelism": f"frame-parallel x{world} (no collective)",
                       "l2_hygiene": f"inputs larger than L2: {B} distinct frames + pyramids{' + outputs' if decode else ''} = "
                                     f"{B * ((2 if decode else 1) * lay.frame_bytes + lay.total_bytes) / 1e6:.0f} MB per step",
                       "step": "forward + inverse pyramid of every frame" if decode else "forward pyramid of every frame",
                       "roundtrip_psnr_db": None if roundtrip_psnr is None else round(float(roundtrip_psnr), 2)},
            "roofline": {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak, "unit": "GB/s",
                         "frac": dom["frac"],
                         "traffic": ncu_traffic_per_launch(traffic_csv) if (B == 16 and CFG["fmt"] == "YUYV") else None,
                         "traffic_source": f"profiles/{traffic_csv} (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum, "
                                           "one launch of 16 4K YUY2 frames)",
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"],
                         "kernel_ms": dom["kernel_ms"], "levels": levels},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="yuv422", choices=sorted(CONFIGS), help="BASELINE.json configuration (default: the one the metric is quoted on)")
    ap.add_argument("--batch", type=int, default=0, help="frames per step per GPU (0 = the config's default)")
    ap.add_argument("--e2e-seconds", type=float, default=2.5, help="length of the timed e2e stream")
    ap.add_argument("--pool-slots", type=int, default=8)
    ap.add_argument("--pool-batch", type=int, default=1)
    ap.add_argument("--pool-inflight", type=int, default=64)
    ap.add_argument("--no-numa-bind", action="store_true", help="do not restrict the rank to its GPU's NUMA node")
    ap.add_argument("--ref-budget-s", type=float, default=150.0, help="wall-clock budget of the whole --impl reference run")
    ap.add_argument("--ref-iters", type=int, default=6, help="frames per host thread (at the full thread count) in the CPU baseline")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="CUDA path only: write the last timed step's coefficients (and decoded frames) of rank 0 as "
                         "DIR/<name>.npy, float32; outputs over the 64 MB budget are a fixed seeded sample")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA path; --impl reference has none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    select_config(args.config)
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
