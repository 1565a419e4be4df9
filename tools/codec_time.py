#!/usr/bin/env python
"""Compress / decompress of the RGBA codec with the host coder and the lane-interleaved device coder (DESIGN.md 4.7).

    python tools/codec_time.py --out DIR [--reps 5] [--sweep-reps 3]

Workload: bench.py's -- batch 16, 768 x 512, RGBACodec random init under torch.manual_seed(234), inputs from
bench.synthetic_rgba.  Reports, with the GPU's name and power limit read in the same run:
  * wall time of compress and decompress per format: median over --reps runs after one warm-up, each run ending in a
    device synchronise;
  * CUDA-event time of the device coder's launches: encode (+ pack) of the y and z strings, and the decode launches of
    one decompress (z and the ten slices), events recorded around each launch inside the timed calls;
  * total stream bytes per format, and whether every reconstruction equals the host format's;
  * a lane sweep (1, 8, the default, 128 lanes): size against time.
Writes DIR/codec_time.json and prints the same JSON.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
import mwa_b200  # noqa: E402

entropy = importlib.import_module(mwa_b200.PACKAGE_NAME + ".entropy")


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = out
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


class LaunchEvents:
    """CUDA events around every encode (encode + pack) and decode launch of the device coder"""

    def __init__(self):
        self.on, self.encode, self.decode = False, [], []
        enc_launch, dec = entropy.LaneEncoding._launch, entropy.LaneDecoder.decode
        timer = self

        def launch(self_):
            return timer._around(timer.encode, lambda: enc_launch(self_))

        def decode(self_, indexes):
            return timer._around(timer.decode, lambda: dec(self_, indexes))

        entropy.LaneEncoding._launch = launch
        entropy.LaneDecoder.decode = decode

    def _around(self, into, fn):
        if not self.on:
            return fn()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = fn()
        b.record()
        into.append((a, b))
        return r

    def take(self):
        torch.cuda.synchronize()
        enc = sum(a.elapsed_time(b) for a, b in self.encode)
        dec = sum(a.elapsed_time(b) for a, b in self.decode)
        counts = (len(self.encode), len(self.decode))
        self.encode, self.decode = [], []
        return enc, dec, counts


def timed(fn, reps):
    """median wall time (ms) over reps runs, each ending in a device synchronise; returns (median, all, last result)"""
    times, r = [], None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = fn()
        torch.cuda.synchronize()
        times.append(1e3 * (time.perf_counter() - t0))
    return statistics.median(times), times, r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sweep-reps", type=int, default=3)
    ap.add_argument("--out", required=True, help="directory for codec_time.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("codec_time.py measures on a CUDA device; none found")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    res = {"gpu": gpu_info(), "workload": f"batch {bench.BATCH_PER_GPU}, {bench.IMG_W}x{bench.IMG_H}, RGBACodec random init "
                                          "(torch.manual_seed(234)), bench.synthetic_rgba(seed0=0)"}
    torch.manual_seed(234)
    net = mwa_b200.RGBACodec().eval().to(dev)
    rgba = bench.synthetic_rgba(bench.BATCH_PER_GPU, seed0=0).to(dev)
    image, alpha = rgba[:, :3].contiguous(), rgba[:, 3:4].contiguous()
    events = LaunchEvents()

    def run(coder, lanes, reps):
        with torch.no_grad():
            comp = lambda: net.compress(image, alpha, coder=coder, lanes=lanes)   # noqa: E731
            out = comp()                                                            # warm-up
            net.decompress(out["strings"], out["shape"], alpha)
            events.on = True
            t_c, all_c, out = timed(comp, reps)
            enc_ms, _, (n_enc, _) = events.take()
            t_d, all_d, rec = timed(lambda: net.decompress(out["strings"], out["shape"], alpha)["x_hat"], reps)
            _, dec_ms, (_, n_dec) = events.take()
            events.on = False
        r = {"compress_ms": t_c, "compress_runs_ms": all_c, "decompress_ms": t_d, "decompress_runs_ms": all_d,
             "bytes": {"y": sum(map(len, out["strings"][0])), "z": sum(map(len, out["strings"][1]))}}
        r["bytes"]["total"] = r["bytes"]["y"] + r["bytes"]["z"]
        r["bpp"] = 8 * r["bytes"]["total"] / (image.shape[0] * image.shape[2] * image.shape[3])
        if coder == "device":
            r["lanes"] = {"y": len(entropy.parse_lanes(out["strings"][0][0])), "z": len(entropy.parse_lanes(out["strings"][1][0]))}
            r["encode_launches_event_ms"] = enc_ms / reps
            r["decode_launches_event_ms"] = dec_ms / reps
            r["launches_per_call"] = {"encode": n_enc // reps, "decode": n_dec // reps}
        return r, rec

    host, rec_host = run("host", None, args.reps)
    device, rec_dev = run("device", None, args.reps)
    device["x_hat_equals_host_format"] = bool(torch.equal(rec_dev, rec_host))
    res["host"], res["device"] = host, device
    res["speedup"] = {"compress": host["compress_ms"] / device["compress_ms"],
                      "decompress": host["decompress_ms"] / device["decompress_ms"]}
    sweep = []
    for lanes in (1, 8, None, 128):                       # None: entropy.default_lanes per message
        r, rec = run("device", lanes, args.sweep_reps)
        sweep.append({"lanes_arg": lanes, "lanes": r["lanes"], "bytes": r["bytes"]["total"],
                      "overhead_vs_host_bytes": r["bytes"]["total"] - host["bytes"]["total"],
                      "compress_ms": r["compress_ms"], "decompress_ms": r["decompress_ms"],
                      "encode_launches_event_ms": r["encode_launches_event_ms"],
                      "decode_launches_event_ms": r["decode_launches_event_ms"],
                      "x_hat_equals_host_format": bool(torch.equal(rec, rec_host))})
    res["lane_sweep"] = sweep
    res["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "codec_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
