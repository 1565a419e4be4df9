#!/usr/bin/env python
"""8- or 16-bit RGBA ingest / egress (csrc/rgba8.cu, DESIGN.md 4.8): kernel time, codec wall time against the fp32-plane
calls, and the host-to-device copy of uint8 / uint16 against fp32.

    python tools/rgba8_time.py --out DIR [--bits 8|16] [--launches 50] [--reps 5]

Reports, with the GPU's name and power limit read in the same run:
  * kernel time of rgba{bits}_ingest (RGBA and alpha-only) and rgba{bits}_egress at batch 16 x 768x512 (bench.py's
    workload) and at
    batch 1 x 2160x3840: CUDA events around each of --launches launches, a 512 MiB buffer written between launches so that
    no launch finds its data in the 126 MB L2; algorithmic bytes per launch (integer samples read / written + fp32 planes
    read / written, the egress reading only the H x W crop of x_hat) and GB/s, against the data-sheet HBM peak (7.7 TB/s,
    HGX B200 per GPU) and against a device-to-device copy measured in the same run;
  * wall time (median of --reps runs after a warm-up, each ending in a device synchronise) of compress_rgba8 /
    decompress_rgba8 (and, with --bits 16, compress_rgba16 / decompress_rgba16 on 257 times the same bytes) and of
    compress / decompress on the same fp32 planes, host and device coder, bench workload, RGBACodec random init under
    torch.manual_seed(234);
  * host-to-device copy of the bench batch from pinned memory: uint8 / uint16 (B, H, W, 4) against fp32 (B, 4, H, W).
Writes DIR/rgba{bits}_time.json and prints the same JSON.

    python tools/rgba8_time.py --tiled --parent-lib PARENT.so --out DIR [--launches 50] [--reps 3]

measures the tiled path instead (DESIGN.md 4.8, "Tiles") and writes DIR/rgba_tiled_time.json:
  * the untiled kernels (rgba8 / rgba16 ingest RGBA, ingest alpha, egress) of this build against those of PARENT.so, the
    library of the commit before the tile kernels, built into a scratch directory (e.g. `git worktree add DIR HEAD~1`, then
    `python -c "import mwa_b200; mwa_b200.build()"` there): launches of the two alternate, one timed pair at a time, at
    the workloads above;
  * the tile kernels on a chunk (2 tiles of 4096 x 4096) of a 1 x 8192 x 8192 image, 8- and 16-bit, with algorithmic
    bytes and GB/s;
  * compress_tiled / decompress_tiled wall time at 1 x 8192 x 8192, both coders, with the chunk count and
    torch.cuda.max_memory_allocated of each call;
  * at 1 x 4096 x 4096, untiled against tile = 2048: string bytes and wall time.  The model is randomly initialised
    (torch.manual_seed(234)), so the bytes show the size of the tiling overhead, not a rate the trained model reaches.
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


def random_samples(shape, bits, g, dev):
    """uniform uint8 / uint16 samples (16-bit ones drawn as int16: uint16 has no CUDA randint)"""
    if bits == 8:
        return torch.randint(0, 256, shape, generator=g, device=dev, dtype=torch.uint8)
    return torch.randint(-2 ** 15, 2 ** 15, shape, generator=g, device=dev, dtype=torch.int16).view(torch.uint16)


def alpha_of(rgba):
    """the alpha channel, contiguous, through a signed view for uint16"""
    s = rgba.view(torch.int16) if rgba.dtype == torch.uint16 else rgba
    return s[..., 3].contiguous().view(rgba.dtype)


def alternated(fns, launches, flush):
    """per-launch CUDA-event times (ms) of each fn, launched in turn, L2 overwritten before each launch"""
    for fn in fns:
        fn()
    torch.cuda.synchronize()
    pairs = [[] for _ in fns]
    for _ in range(launches):
        for k, fn in enumerate(fns):
            flush.add_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            pairs[k].append((a, b))
    torch.cuda.synchronize()
    return [[a.elapsed_time(b) for a, b in p] for p in pairs]


def tiled(args, dev):
    import ctypes
    res = {"gpu": gpu_info(), "hbm_peak": f"{HBM_PEAK_GBPS:.0f} GB/s (NVIDIA HGX B200 data sheet, per GPU)"}
    lib = mwa_b200._abi.load()
    parent = ctypes.CDLL(os.path.abspath(args.parent_lib))
    for name in ("rgba8_ingest", "rgba8_egress", "rgba16_ingest", "rgba16_egress"):
        fn = getattr(parent, name)
        fn.restype, fn.argtypes = ctypes.c_int, getattr(lib, name).argtypes
    flush = torch.zeros(128 * 2 ** 20, dtype=torch.float32, device=dev)            # 512 MiB
    src = torch.ones(256 * 2 ** 20, dtype=torch.float32, device=dev)
    dst = torch.empty_like(src)
    ct = event_times(lambda: dst.copy_(src), args.launches, flush)
    copy_gbps = 2 * src.numel() * 4 / (statistics.median(ct) * 1e-3) / 1e9
    res["copy_1GiB"] = {"median_us": 1e3 * statistics.median(ct), "bytes": 2 * src.numel() * 4, "GBps": copy_gbps}
    del src, dst

    def run(fn, *a):
        mwa_b200._abi.check(fn(*a, mwa_b200._abi.stream_handle()), fn.__name__)

    # the untiled kernels, this build against the parent's, alternated
    untiled = {}
    for wl, (B, H, W) in {"bench_16x768x512": (bench.BATCH_PER_GPU, bench.IMG_H, bench.IMG_W),
                          "1x3840x2160": (1, 2160, 3840)}.items():
        for bits in (8, 16):
            g = torch.Generator(device=dev).manual_seed(1)
            rgba = random_samples((B, H, W, 4), bits, g, dev)
            a = alpha_of(rgba)
            Hp, Wp = padded(H), padded(W)
            image = torch.empty(B, 3, Hp, Wp, device=dev)
            alpha = torch.empty(B, 1, Hp, Wp, device=dev)
            x_hat = torch.rand(B, 3, Hp, Wp, generator=g, device=dev)
            out = torch.empty_like(rgba)
            calls = {"ingest_rgba": lambda L: run(getattr(L, f"rgba{bits}_ingest"), rgba.data_ptr(), image.data_ptr(),
                                                  alpha.data_ptr(), B, H, W, 4),
                     "ingest_alpha": lambda L: run(getattr(L, f"rgba{bits}_ingest"), a.data_ptr(), None, alpha.data_ptr(),
                                                   B, H, W, 1),
                     "egress": lambda L: run(getattr(L, f"rgba{bits}_egress"), x_hat.data_ptr(), a.data_ptr(),
                                             out.data_ptr(), B, H, W)}
            for kname, call in calls.items():
                this_t, parent_t = alternated([lambda: call(lib), lambda: call(parent)], args.launches, flush)
                untiled[f"{wl}/rgba{bits}/{kname}"] = {
                    k: {"median_us": 1e3 * statistics.median(t), "min_us": 1e3 * min(t), "max_us": 1e3 * max(t),
                        "q1_us": 1e3 * statistics.quantiles(t, n=4)[0], "q3_us": 1e3 * statistics.quantiles(t, n=4)[2]}
                    for k, t in (("this", this_t), ("parent", parent_t))}
            del rgba, a, image, alpha, x_hat, out
    res["untiled_kernels_this_vs_parent"] = untiled

    # the tile kernels on one chunk of an 8192 x 8192 image
    H = W = 8192
    Th, Tw, ty, tx = mwa_b200.rgba8.tile_grid(H, W, 4096)
    count = mwa_b200.rgba8.chunk_tiles(Th, Tw)
    kern = {"H": H, "W": W, "tile": (Th, Tw), "grid": (ty, tx), "count": count}
    px = count * Th * Tw                        # every pixel of these tiles lies in the image
    for bits in (8, 16):
        sb = bits // 8
        g = torch.Generator(device=dev).manual_seed(2)
        rgba = random_samples((1, H, W, 4), bits, g, dev)
        a = alpha_of(rgba)
        x_hat = torch.rand(count, 3, Th, Tw, generator=g, device=dev)
        out = torch.empty_like(rgba)
        r = mwa_b200.rgba8
        for kname, fn, nbytes in (("ingest_rgba", lambda: r.ingest_tiles(rgba, (Th, Tw), 0, count), 4 * sb * px + 16 * px),
                                  ("ingest_alpha", lambda: r.ingest_tiles(a[..., None], (Th, Tw), 0, count),
                                   sb * px + 4 * px),
                                  ("egress", lambda: r.egress_tiles(x_hat, a, out, 0), 12 * px + sb * px + 4 * sb * px)):
            kern[f"rgba{bits}/{kname}"] = summary(event_times(fn, args.launches, flush), nbytes, copy_gbps)
        del rgba, a, x_hat, out
    res["tile_kernels_8192"] = kern
    del flush

    # the codec
    torch.manual_seed(234)
    net = mwa_b200.RGBACodec().eval().to(dev)
    g = torch.Generator().manual_seed(3)

    def picture(H, W):
        """smooth colour in 16 x 16 blocks + noise, alpha 0 on ~25 % of the blocks (uint8 on the device)"""
        small = torch.rand(1, 4, -(-H // 16), -(-W // 16), generator=g)
        small[:, 3] = small[:, 3] * (small[:, 3] > 0.25)
        big = torch.nn.functional.interpolate(small, scale_factor=16, mode="bilinear")[..., :H, :W]
        big = (big + 0.03 * torch.randn(big.shape, generator=g)).clamp(0, 1)
        big[:, 3] *= big[:, 3] > 0.2
        return (big * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous().to(dev)

    def measured(fn):
        fn()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        med, runs, out = timed(fn, args.reps)
        return {"median_ms": med, "runs_ms": runs, "max_memory_allocated_GB": torch.cuda.max_memory_allocated() / 1e9}, out

    codec = {"model": "RGBACodec, random init under torch.manual_seed(234)",
             "free_and_total_GB_at_start": [v / 1e9 for v in torch.cuda.mem_get_info()]}
    t = picture(8192, 8192)
    a8 = alpha_of(t)
    with torch.no_grad():
        for coder in ("host", "device"):
            c, out = measured(lambda: net.compress_tiled(t, coder=coder))
            d, rec = measured(lambda: net.decompress_tiled(out["strings"], out["shape"], a8))
            n = len(out["strings"][0])
            codec[f"1x8192x8192/{coder}"] = {
                "grid": out["grid"], "shape": tuple(out["shape"]), "tiles": n,
                "chunks": -(-n // mwa_b200.rgba8.chunk_tiles(64 * out["shape"][0], 64 * out["shape"][1])),
                "bytes": sum(map(len, out["strings"][0])) + sum(map(len, out["strings"][1])),
                "compress_tiled": c, "decompress_tiled": d,
                "alpha_copied": bool(torch.equal(rec[..., 3], a8))}
        del t, a8, rec
        t = picture(4096, 4096)
        a8 = alpha_of(t)
        for coder in ("host", "device"):
            for label, comp, decomp in (
                    ("untiled", lambda: net.compress_rgba8(t, coder=coder),
                     lambda o: net.decompress_rgba8(o["strings"], o["shape"], a8)),
                    ("tile_2048", lambda: net.compress_tiled(t, 2048, coder=coder),
                     lambda o: net.decompress_tiled(o["strings"], o["shape"], a8))):
                c, out = measured(comp)
                d, rec = measured(lambda: decomp(out))
                err = (rec[..., :3].float() - t[..., :3].float()) * (a8[..., None] > 0)
                codec[f"1x4096x4096/{coder}/{label}"] = {
                    "tiles": len(out["strings"][0]),
                    "bytes": sum(map(len, out["strings"][0])) + sum(map(len, out["strings"][1])),
                    "compress": c, "decompress": d, "rgb_mse_opaque": float(err.square().sum() / (a8 > 0).sum() / 3)}
    res["codec"] = codec
    res["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "rgba_tiled_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--bits", type=int, choices=(8, 16), default=8, help="sample depth of the timed kernels")
    ap.add_argument("--tiled", action="store_true", help="measure the tiled path (rgba_tiled_time.json)")
    ap.add_argument("--parent-lib", help="with --tiled: the previous commit's libmwa_b200.so, for the untiled kernels")
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("rgba8_time.py measures on a CUDA device; none found")
    if args.tiled:
        if not args.parent_lib:
            sys.exit("--tiled needs --parent-lib")
        return tiled(args, torch.device("cuda:0"))
    dev = torch.device("cuda:0")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    bits, sb = args.bits, args.bits // 8                                        # sample bytes
    ingest, egress = getattr(mwa_b200, f"rgba{bits}_ingest"), getattr(mwa_b200, f"rgba{bits}_egress")
    res = {"gpu": gpu_info(), "bits": bits, "hbm_peak": f"{HBM_PEAK_GBPS:.0f} GB/s (NVIDIA HGX B200 data sheet, per GPU)"}
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
        if bits == 8:
            rgba = torch.randint(0, 256, (B, H, W, 4), generator=g, device=dev, dtype=torch.uint8)
        else:                                   # uniform 16-bit patterns, drawn as int16 (uint16 has no CUDA randint)
            rgba = torch.randint(-2 ** 15, 2 ** 15, (B, H, W, 4), generator=g, device=dev, dtype=torch.int16).view(torch.uint16)
        a8 = rgba[..., 3].contiguous() if bits == 8 else rgba.view(torch.int16)[..., 3].contiguous().view(torch.uint16)
        Hp, Wp = padded(H), padded(W)
        x_hat = torch.rand(B, 3, Hp, Wp, generator=g, device=dev)
        px, ppx = B * H * W, B * Hp * Wp
        k = {"B": B, "H": H, "W": W, "Hp": Hp, "Wp": Wp}
        k["ingest_rgba"] = summary(event_times(lambda: ingest(rgba), args.launches, flush),
                                   4 * sb * px + 4 * 4 * ppx, copy_gbps)
        k["ingest_alpha"] = summary(event_times(lambda: ingest(a8[..., None]), args.launches, flush),
                                    sb * px + 4 * ppx, copy_gbps)
        k["egress"] = summary(event_times(lambda: egress(x_hat, a8), args.launches, flush),
                              3 * 4 * px + sb * px + 4 * sb * px, copy_gbps)
        kernels[name] = k
        del rgba, a8, x_hat
    res["kernels"] = kernels
    del flush

    # codec wall time on the bench workload
    torch.manual_seed(234)
    net = mwa_b200.RGBACodec().eval().to(dev)
    planes = bench.synthetic_rgba(bench.BATCH_PER_GPU, seed0=0)
    rgba8 = (planes.permute(0, 2, 3, 1) * 255).round().to(torch.uint8).contiguous()
    depths = {8: rgba8}
    if bits == 16:
        depths[16] = (rgba8.to(torch.int32) * 257).to(torch.uint16)       # the same planes at 16 bits (DESIGN.md 4.8)
    on_dev = {d: t.to(dev) for d, t in depths.items()}
    alphas = {d: t[..., 3].contiguous().to(dev) for d, t in depths.items()}
    image, alpha, _ = mwa_b200.rgba8_ingest(on_dev[8])            # the same planes compress_rgba8 codes
    wall = {"workload": f"batch {bench.BATCH_PER_GPU}, {bench.IMG_W}x{bench.IMG_H}, bench.synthetic_rgba(seed0=0) as uint8"
                        f"{' (and 257 times it as uint16)' if bits == 16 else ''}, RGBACodec random init "
                        "(torch.manual_seed(234)), inputs on the device"}
    with torch.no_grad():
        for coder in ("host", "device"):
            r = {}
            comp = {d: getattr(net, f"compress_rgba{d}") for d in depths}
            decomp = {d: getattr(net, f"decompress_rgba{d}") for d in depths}
            out = net.compress(image, alpha, coder=coder)
            net.decompress(out["strings"], out["shape"], alpha)
            for d in depths:
                o = comp[d](on_dev[d], coder=coder)
                decomp[d](o["strings"], o["shape"], alphas[d])
            r["compress_ms"], r["compress_runs_ms"], out = timed(lambda: net.compress(image, alpha, coder=coder), args.reps)
            r["decompress_ms"], r["decompress_runs_ms"], rec = timed(
                lambda: net.decompress(out["strings"], out["shape"], alpha)["x_hat"], args.reps)
            for d in depths:
                r[f"compress_rgba{d}_ms"], r[f"compress_rgba{d}_runs_ms"], o = timed(
                    lambda: comp[d](on_dev[d], coder=coder), args.reps)
                r[f"decompress_rgba{d}_ms"], r[f"decompress_rgba{d}_runs_ms"], rec_d = timed(
                    lambda: decomp[d](o["strings"], o["shape"], alphas[d]), args.reps)
                suffix = "" if d == 8 else f"_rgba{d}"
                r["strings_equal" + suffix] = o["strings"] == out["strings"]
                # compared on the CPU in int32: torch has no CUDA comparison for uint16
                want = (rec[:, :, :bench.IMG_H, :bench.IMG_W] * (2 ** d - 1)).round().to(torch.int32).permute(0, 2, 3, 1)
                got = rec_d[..., :3].cpu().to(torch.int32)
                opaque = alphas[d].cpu().to(torch.int32)[..., None] > 0
                r[f"rgb_equals_quantised_decompress{suffix}"] = bool(torch.equal(got, want.cpu() * opaque))
            wall[coder] = r
    res["codec_wall"] = wall

    # host -> device copy from pinned memory
    h8 = depths[bits].pin_memory()
    h32 = planes.contiguous().pin_memory()
    d8, d32 = torch.empty_like(h8, device=dev), torch.empty_like(h32, device=dev)
    copies = {}
    for name, (h, d) in {f"uint{bits}_BHW4": (h8, d8), "fp32_B4HW": (h32, d32)}.items():
        t = event_times(lambda: d.copy_(h, non_blocking=True), 20, torch.zeros(1, device=dev))
        med = statistics.median(t)
        copies[name] = {"bytes": h.numel() * h.element_size(), "median_ms": med,
                        "GBps": h.numel() * h.element_size() / (med * 1e-3) / 1e9}
    res["h2d_pinned"] = copies
    res["gpu_after"] = gpu_info()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, f"rgba{bits}_time.json"), "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
