#!/usr/bin/env python
"""8-bit RGBA ingest / egress (csrc/rgba8.cu, DESIGN.md 4.8): kernel time, codec wall time against the fp32-plane calls, and
the host-to-device copy of uint8 against fp32.

    python tools/rgba8_time.py --out DIR [--launches 50] [--reps 5]

Reports, with the GPU's name and power limit read in the same run:
  * kernel time of rgba8_ingest (RGBA and alpha-only) and rgba8_egress at batch 16 x 768x512 (bench.py's workload) and at
    batch 1 x 2160x3840: CUDA events around each of --launches launches, a 512 MiB buffer written between launches so that
    no launch finds its data in the 126 MB L2; algorithmic bytes per launch (uint8 read / written + fp32 planes read /
    written, the egress reading only the H x W crop of x_hat) and GB/s, against the data-sheet HBM peak (7.7 TB/s, HGX B200
    per GPU) and against a device-to-device copy measured in the same run;
  * wall time (median of --reps runs after a warm-up, each ending in a device synchronise) of compress_rgba8 /
    decompress_rgba8 and of compress / decompress on the same fp32 planes, host and device coder, bench workload, RGBACodec
    random init under torch.manual_seed(234);
  * host-to-device copy of the bench batch from pinned memory: uint8 (B, H, W, 4) against fp32 (B, 4, H, W).
Writes DIR/rgba8_time.json and prints the same JSON.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench  # noqa: E402
import mwa_b200  # noqa: E402
from codec_time import gpu_info, timed  # noqa: E402

HBM_PEAK_GBPS = 7700.0          # NVIDIA HGX B200 data sheet, per GPU


def padded(n):
    return -(-n // 64) * 64


def event_times(fn, launches, flush):
    """per-launch CUDA-event times (ms), L2 overwritten before each launch"""
    fn()
    torch.cuda.synchronize()
    pairs = []
    for _ in range(launches):
        flush.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        pairs.append((a, b))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in pairs]


def summary(times, nbytes, copy_gbps):
    med = statistics.median(times)
    gbps = nbytes / (med * 1e-3) / 1e9
    return {"median_us": 1e3 * med, "min_us": 1e3 * min(times), "max_us": 1e3 * max(times), "launches": len(times),
            "bytes": nbytes, "GBps": gbps, "of_hbm_peak_datasheet": gbps / HBM_PEAK_GBPS,
            "of_measured_copy": gbps / copy_gbps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", required=True, help="directory for rgba8_time.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rgba8_time.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"gpu": gpu_info(), "hbm_peak": f"{HBM_PEAK_GBPS:.0f} GB/s (NVIDIA HGX B200 data sheet, per GPU)"}
    flush = torch.zeros(128 * 2 ** 20, dtype=torch.float32, device=dev)            # 512 MiB

    # device-to-device copy in the same run: the rate an HBM-bound pass of this size can reach here
    src = torch.ones(256 * 2 ** 20, dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    ct = event_times(lambda: dst.copy_(src), args.launches, flush)
    copy_gbps = 2 * src.numel() * 4 / (statistics.median(ct) * 1e-3) / 1e9
    res["copy_1GiB"] = {"median_us": 1e3 * statistics.median(ct), "bytes": 2 * src.numel() * 4, "GBps": copy_gbps}
    del src, dst

    kernels = {}
    for name, (B, H, W) in {"bench_16x768x512": (bench.BATCH_PER_GPU, bench.IMG_H, bench.IMG_W),
                            "1x3840x2160": (1, 2160, 3840)}.items():
        g = torch.Generator(device=dev).manual_seed(1)
        rgba = torch.randint(0, 256, (B, H, W, 4), generator=g, device=dev, dtype=torch.uint8)
        a8 = rgba[..., 3].contiguous()
        Hp, Wp = padded(H), padded(W)
        x_hat = torch.rand(B, 3, Hp, Wp, generator=g, device=dev)
        px, ppx = B * H * W, B * Hp * Wp
        k = {"B": B, "H": H, "W": W, "Hp": Hp, "Wp": Wp}
        k["ingest_rgba"] = summary(event_times(lambda: mwa_b200.rgba8_ingest(rgba), args.launches, flush),
                                   4 * px + 4 * 4 * ppx, copy_gbps)
        k["ingest_alpha"] = summary(event_times(lambda: mwa_b200.rgba8_ingest(a8[..., None]), args.launches, flush),
                                    px + 4 * ppx, copy_gbps)
        k["egress"] = summary(event_times(lambda: mwa_b200.rgba8_egress(x_hat, a8), args.launches, flush),
                              3 * 4 * px + px + 4 * px, copy_gbps)
        kernels[name] = k
        del rgba, a8, x_hat
    res["kernels"] = kernels
    del flush

    # codec wall time on the bench workload
    torch.manual_seed(234)
    net = mwa_b200.RGBACodec().eval().to(dev)
    planes = bench.synthetic_rgba(bench.BATCH_PER_GPU, seed0=0)
    rgba8 = (planes.permute(0, 2, 3, 1) * 255).round().to(torch.uint8).contiguous()
    rgba8_dev = rgba8.to(dev)
    image, alpha, _ = mwa_b200.rgba8_ingest(rgba8_dev)           # the same planes compress_rgba8 codes
    a8 = rgba8_dev[..., 3].contiguous()
    wall = {"workload": f"batch {bench.BATCH_PER_GPU}, {bench.IMG_W}x{bench.IMG_H}, bench.synthetic_rgba(seed0=0) as uint8, "
                        "RGBACodec random init (torch.manual_seed(234)), inputs on the device"}
    with torch.no_grad():
        for coder in ("host", "device"):
            r = {}
            out8 = net.compress_rgba8(rgba8_dev, coder=coder)
            out = net.compress(image, alpha, coder=coder)
            net.decompress_rgba8(out8["strings"], out8["shape"], a8)
            net.decompress(out["strings"], out["shape"], alpha)
            r["compress_rgba8_ms"], r["compress_rgba8_runs_ms"], out8 = timed(
                lambda: net.compress_rgba8(rgba8_dev, coder=coder), args.reps)
            r["compress_ms"], r["compress_runs_ms"], out = timed(lambda: net.compress(image, alpha, coder=coder), args.reps)
            r["decompress_rgba8_ms"], r["decompress_rgba8_runs_ms"], rec8 = timed(
                lambda: net.decompress_rgba8(out8["strings"], out8["shape"], a8), args.reps)
            r["decompress_ms"], r["decompress_runs_ms"], rec = timed(
                lambda: net.decompress(out["strings"], out["shape"], alpha)["x_hat"], args.reps)
            r["strings_equal"] = out8["strings"] == out["strings"]
            want = (rec[:, :, :bench.IMG_H, :bench.IMG_W] * 255).round().to(torch.uint8).permute(0, 2, 3, 1)
            r["rgb_equals_quantised_decompress"] = bool(torch.equal(rec8[..., :3], want * (a8[..., None] > 0)))
            wall[coder] = r
    res["codec_wall"] = wall

    # host -> device copy from pinned memory
    h8 = rgba8.pin_memory()
    h32 = planes.contiguous().pin_memory()
    d8, d32 = torch.empty_like(h8, device=dev), torch.empty_like(h32, device=dev)
    copies = {}
    for name, (h, d) in {"uint8_BHW4": (h8, d8), "fp32_B4HW": (h32, d32)}.items():
        t = event_times(lambda: d.copy_(h, non_blocking=True), 20, torch.zeros(1, device=dev))
        med = statistics.median(t)
        copies[name] = {"bytes": h.numel() * h.element_size(), "median_ms": med,
                        "GBps": h.numel() * h.element_size() / (med * 1e-3) / 1e9}
    res["h2d_pinned"] = copies
    res["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "rgba8_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
