#!/usr/bin/env python
"""Masked MS-SSIM as a loss (csrc/msssim.cu, DESIGN.md 4.5): kernel time of the forward and of the backward against the
oracle's torch expressions run in fp32 on the same device under autograd.

    python tools/msssim_time.py --out DIR [--launches 30]

Workloads: the training crop (8 x 3 x 256x256) and bench.py's batch (16 x 3 x 768x512), X = bench.synthetic_rgba's colour
planes, Y = X + noise, the mask = its alpha.  For each, with the GPU's name and power limit read in the same run:
  * forward (no grad), forward + backward, and the backward alone (ms_ssim_level_backward x 5 plus the torch tail): CUDA
    events around each of --launches passes after a warm-up, a 512 MiB buffer written before every pass so that no pass
    finds its data in the 126 MB L2;
  * the five backward launches alone, from CUDA events around each launch;
  * algorithmic bytes of the backward launches (X, Y, mask read, dX, dY written, the coarser dX, dY read once) and GB/s
    against the data-sheet HBM peak (7.7 TB/s, HGX B200 per GPU);
  * the same forward + backward through oracle/ref_model.masked_ms_ssim in fp32 on the device.
Writes DIR/msssim_time.json and prints the same JSON.
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
from codec_time import gpu_info  # noqa: E402
from oracle import ref_model as M  # noqa: E402

HBM_PEAK_GBPS = 7700.0          # NVIDIA HGX B200 data sheet, per GPU
WORKLOADS = {"train_8x3x256x256": (8, 256, 256), "bench_16x3x768x512": (bench.BATCH_PER_GPU, bench.IMG_H, bench.IMG_W)}


def inputs(B, H, W, dev):
    old = bench.IMG_H, bench.IMG_W
    bench.IMG_H, bench.IMG_W = H, W
    try:
        rgba = bench.synthetic_rgba(B, seed0=0)
    finally:
        bench.IMG_H, bench.IMG_W = old
    g = torch.Generator().manual_seed(1)
    X = rgba[:, :3].contiguous()
    Y = (X + 0.05 * torch.randn(X.shape, generator=g)).clamp(0, 1)
    return X.to(dev), Y.to(dev), rgba[:, 3:4].contiguous().to(dev)


def backward_bytes(B, C, H, W, levels=5):
    """HBM bytes the backward launches must move: per level X, Y, mask read and dX, dY written, plus the coarser level's
    dX, dY read once"""
    total = 0
    for lvl in range(levels):
        total += 4 * (2 * B * C * H * W + B * H * W + 2 * B * C * H * W)
        Hp, Wp = (H + 2 * (H % 2) - 2) // 2 + 1, (W + 2 * (W % 2) - 2) // 2 + 1
        if lvl < levels - 1:
            total += 4 * 2 * B * C * Hp * Wp
        H, W = Hp, Wp
    return total


def passes(fn, launches, flush, setup=None):
    """per-pass CUDA-event times (ms) of fn, L2 overwritten and setup() run (untimed) before each pass"""
    for _ in range(2):
        fn(setup() if setup else None)
    torch.cuda.synchronize()
    pairs = []
    for _ in range(launches):
        flush.add_(1)
        arg = setup() if setup else None
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(arg)
        b.record()
        pairs.append((a, b))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in pairs]


def stats(times):
    return {"median_ms": statistics.median(times), "min_ms": min(times), "max_ms": max(times), "passes": len(times)}


class LaunchEvents:
    """CUDA events around every ms_ssim_level_backward call"""

    def __init__(self, lib):
        self.lib, self.real, self.pairs = lib, lib.ms_ssim_level_backward, []

    def __call__(self, *args):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        status = self.real(*args)
        b.record()
        self.pairs.append((a, b))
        return status

    def __enter__(self):
        self.lib.ms_ssim_level_backward = self
        return self

    def __exit__(self, *exc):
        self.lib.ms_ssim_level_backward = self.real
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--out", required=True, help="directory for msssim_time.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("msssim_time.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    lib = mwa_b200._abi.load()
    res = {"gpu": gpu_info(), "hbm_peak": f"{HBM_PEAK_GBPS:.0f} GB/s (NVIDIA HGX B200 data sheet, per GPU)",
           "l2": "a 512 MiB buffer is written before every timed pass"}
    flush = torch.zeros(128 * 2 ** 20, dtype=torch.float32, device=dev)
    out = {}
    for name, (B, H, W) in WORKLOADS.items():
        X, Y, mask = inputs(B, H, W, dev)
        Xg, Yg = X.clone().requires_grad_(True), Y.clone().requires_grad_(True)
        r = {"B": B, "C": 3, "H": H, "W": W}

        def fwd(_):
            with torch.no_grad():
                mwa_b200.masked_ms_ssim(X, Y, mask)

        def fwd_bwd(_):
            Xg.grad = Yg.grad = None
            (1 - mwa_b200.masked_ms_ssim(Xg, Yg, mask)).backward()

        def graph():
            Xg.grad = Yg.grad = None
            return 1 - mwa_b200.masked_ms_ssim(Xg, Yg, mask)

        def oracle(_):
            Xg.grad = Yg.grad = None
            with torch.device(dev):
                (1 - M.masked_ms_ssim(Xg, Yg, mask)).backward()

        r["forward_no_grad"] = stats(passes(fwd, args.launches, flush))
        r["forward_backward"] = stats(passes(fwd_bwd, args.launches, flush))
        r["backward"] = stats(passes(lambda loss: loss.backward(), args.launches, flush, setup=graph))
        # the five backward launches alone
        per_pass = []
        for _ in range(args.launches):
            loss = graph()
            flush.add_(1)
            with LaunchEvents(lib) as ev:
                loss.backward()
            per_pass.append(ev)
        torch.cuda.synchronize()
        kt = [sum(a.elapsed_time(b) for a, b in ev.pairs) for ev in per_pass]
        nbytes = backward_bytes(B, 3, H, W)
        med = statistics.median(kt)
        r["backward_kernels"] = {**stats(kt), "launches_per_pass": len(per_pass[0].pairs), "bytes": nbytes,
                                 "GBps": nbytes / (med * 1e-3) / 1e9,
                                 "of_hbm_peak_datasheet": nbytes / (med * 1e-3) / 1e9 / HBM_PEAK_GBPS}
        r["oracle_fp32_forward_backward"] = stats(passes(oracle, max(5, args.launches // 3), flush))
        r["speedup_forward_backward"] = r["oracle_fp32_forward_backward"]["median_ms"] / r["forward_backward"]["median_ms"]
        # gradients of the two, for the record
        Xg.grad = Yg.grad = None
        (1 - mwa_b200.masked_ms_ssim(Xg, Yg, mask)).backward()
        gd = Xg.grad.clone()
        oracle(None)
        r["dX_max_abs_diff_over_max"] = float((gd - Xg.grad).abs().max() / Xg.grad.abs().max())
        out[name] = r
        del X, Y, mask, Xg, Yg
        torch.cuda.empty_cache()
    res["workloads"] = out
    res["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "msssim_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
