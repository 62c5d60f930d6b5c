"""Timing of the final 4:2:2 inverse level (k_inv_422) per output format: 8-bit YUYV, 16-bit YU64 and 10-bit V210.

Device-resident, 16 x 3840x2160 frames per launch, only level 1 inverted (the levels above are left as a full forward
wrote them), CUDA events on the launching stream.  The formats alternate round by round in one process, so they share
clocks and neighbours; the median round is reported.  Achieved bandwidth = algorithmic bytes (the twelve level-1 bands
read once, 4 bytes per pixel, + the packed output written once) over kernel time, against MEASURED_PEAKS.json hbm_gbs
where present.  The working set of one launch (16 x ~56-66 MB) is far larger than the 126 MB L2.
Also checks, on one frame, that the V210 output is the YU64 output >> 6 wherever a 6-pixel group is complete.

    python tools/inv_out_bench.py [--out FILE]"""
import argparse
import importlib
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception:
        q = torch.cuda.get_device_name(0) + ", power limit unknown"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=3840)
    ap.add_argument("--height", type=int, default=2160)
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None, help="also write the report to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("inv_out_bench: no CUDA device")
    pkg = importlib.import_module("cineform-sdk_b200")
    import bench
    w, h, n = a.width, a.height, a.batch
    torch.cuda.init()
    ctx = pkg.Context(0)
    desc = pkg.FrameDesc(w, h, pkg.PIXEL_YUYV)
    quant = pkg.quant_for_quality(desc, 4)
    codec = pkg.Codec(ctx, desc, 1)
    lay = codec.layout
    stream = torch.cuda.ExternalStream(ctx.stream)
    # output format -> (CFB pixel format, pitch = bytes per row)
    fmts = {"YUYV": (pkg.PIXEL_YUYV, 2 * w), "YU64": (pkg.PIXEL_YU64, 4 * w), "V210": (pkg.PIXEL_V210, pkg.v210_pitch(w))}
    frames = bench.synthetic_frames(n, w, h)
    with torch.cuda.stream(stream):
        d_frames = [torch.from_numpy(np.ascontiguousarray(f).reshape(-1)).cuda() for f in frames]
        d_pyr = [torch.zeros(lay.total_bytes, dtype=torch.uint8, device="cuda") for _ in range(n)]
        d_out = [torch.zeros(4 * w * h, dtype=torch.uint8, device="cuda") for _ in range(n)]
    fp, pp, op = [t.data_ptr() for t in d_frames], [t.data_ptr() for t in d_pyr], [t.data_ptr() for t in d_out]
    codec.forward_device(fp, lay.frame_pitch, quant, pp)          # every band of every frame holds real coefficients
    ctx.synchronize()
    codec.set_level_mask(0, 1)                                    # invert level 1 only: one k_inv_422 launch per call
    P = sum(lay.band[c][0][0].width * lay.band[c][0][0].height * 4 for c in range(lay.num_channels))
    band_bytes = 2 * P

    def run(name):
        codec.inverse_device(pp, quant, fmts[name][0], op, fmts[name][1])

    for name in fmts:
        for _ in range(5):
            run(name)
    ctx.synchronize()
    times = {name: [] for name in fmts}
    for _ in range(a.rounds):
        for name in fmts:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(a.iters):
                run(name)
            e1.record(stream)
            ctx.synchronize()
            times[name].append(e0.elapsed_time(e1) * 1e3 / a.iters)

    # V210 == YU64 >> 6 on the complete groups of frame 0 (the level-1 input is identical between the two calls)
    outs = {}
    for name in ("YU64", "V210"):
        run(name)
        ctx.synchronize()
        outs[name] = d_out[0][:fmts[name][1] * h].cpu().numpy()
    y16 = outs["YU64"].view(np.uint16).reshape(h, 2 * w)
    g = w // 6
    y, c1, c3 = [(v >> 6).astype(np.uint32) for v in (y16[:, 0::2], y16[:, 1::4], y16[:, 3::4])]
    comp = np.zeros((h, 12 * g), np.uint32)
    comp[:, 0::4], comp[:, 1::4], comp[:, 2::4], comp[:, 3::4] = c3[:, :3 * g], y[:, 0:6 * g:2], c1[:, :3 * g], y[:, 1:6 * g:2]
    v210 = outs["V210"].view(np.uint32).reshape(h, -1)[:, :4 * g]
    same = bool(np.array_equal(v210, comp[:, 0::3] | (comp[:, 1::3] << 10) | (comp[:, 2::3] << 20)))

    peak, peak_src = bench.peaks()
    lines = [f"k_inv_422 (level 1 only), {n} x {w}x{h} per launch, {a.iters} launches x {a.rounds} alternating rounds, "
             f"CUDA events; GPU: {gpu_identity()}; peak {peak:.0f} GB/s {peak_src}"]
    for name, (_, pitch) in fmts.items():
        out_bytes = pitch * h
        us = statistics.median(times[name])
        gbs = (band_bytes + out_bytes) * n / (us * 1e-6) / 1e9
        lines.append(f"{name}: median {us:.1f} us per launch (min {min(times[name]):.1f}, max {max(times[name]):.1f}), "
                     f"output {out_bytes / 1e6:.1f} MB/frame + bands {band_bytes / 1e6:.1f} MB/frame -> {gbs:.0f} GB/s, "
                     f"{gbs / peak:.3f} of peak")
    lines.append(f"V210 complete groups == YU64 >> 6 on frame 0: {same}")
    report = "\n".join(lines)
    print(report, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(report + "\n")
    if not same:
        sys.exit(1)


if __name__ == "__main__":
    main()
