#!/usr/bin/env python
"""Kernel micro-benchmarks (development tool, run on the B200 box):
times each hot-path kernel alone with CUDA events at the BASELINE config-2 shapes, prints the roofline
fraction, and cross-checks the default kernels against the fp32 SIMT kernels on the same inputs.

    python tools/kbench.py [gdn] [attn] [round] [--iters 20]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import mwa_b200 as pkg  # noqa: E402

PEAKS = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(
    os.path.join(ROOT, "MEASURED_PEAKS.json")) else {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0}


def timeit(fn, iters, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        flush.add_(1.0)                       # 512 MB write: evicts L2 between timed launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def bench_gdn(args, dev, flush):
    g = torch.Generator(device=dev).manual_seed(0)
    for inverse in (False, True):
        m = pkg.GDN(192, inverse=inverse)
        with torch.no_grad():
            m.gamma.add_(torch.rand(192, 192) * 0.02)
            m.beta.mul_(0.5 + torch.rand(192))
        m = m.to(dev)
        for (B, H, W) in ((16, 256, 384), (16, 128, 192), (16, 64, 96)):
            x = torch.randn(B, 192, H, W, device=dev, generator=g) * 2
            res = {}
            for name, algo in (("simt", pkg.ALGO_SIMT), ("tcgen05", pkg.ALGO_TCGEN05)):
                m.algo = algo
                try:
                    with torch.no_grad():
                        y = m(x)
                        med, best = timeit(lambda: m(x), args.iters if name != "simt" else 3, flush)
                except pkg.MwaB200Error as e:
                    print(f"gdn inverse={inverse} {B}x192x{H}x{W} {name}: {e}")
                    continue
                res[name] = y
                gb = x.numel() * 8 / 1e9
                print(f"gdn inverse={int(inverse)} {B}x192x{H}x{W} {name:8s} median {med:8.3f} ms  best {best:8.3f} ms  "
                      f"{gb / med * 1e3:8.1f} GB/s  = {gb / med * 1e3 / PEAKS['hbm_gbs'] * 100:5.1f}% of measured HBM peak",
                      flush=True)
            # channels_last (NHWC) input through the same module
            xcl = x.contiguous(memory_format=torch.channels_last)
            m.algo = pkg.ALGO_TCGEN05
            with torch.no_grad():
                ycl = m(xcl)
                med, best = timeit(lambda: m(xcl), args.iters, flush)
            gb = x.numel() * 8 / 1e9
            print(f"gdn inverse={int(inverse)} {B}x192x{H}x{W} tc-NHWC  median {med:8.3f} ms  best {best:8.3f} ms  "
                  f"{gb / med * 1e3:8.1f} GB/s  = {gb / med * 1e3 / PEAKS['hbm_gbs'] * 100:5.1f}% of measured HBM peak; "
                  f"max |NHWC - NCHW| {(ycl - res['tcgen05']).abs().max().item():.2e}", flush=True)
            if len(res) == 2:
                d = (res["simt"] - res["tcgen05"]).abs()
                rel = d / (res["simt"].abs() + 1e-4 / 1e-3)
                print(f"    tcgen05 vs simt: max abs diff {d.max().item():.3e}, max |d|/(|ref|+0.1) {rel.max().item():.3e}, "
                      f"allclose(1e-3,1e-4) {torch.allclose(res['tcgen05'], res['simt'], rtol=1e-3, atol=1e-4)}",
                      flush=True)


def bench_attn(args, dev, flush):
    from oracle import golden_cases as G
    from oracle import ref_ops as R
    for (C, heads, ws, s, H, W) in ((192, 8, 8, 4, 128, 192), (192, 6, 8, 4, 128, 192), (80, 8, 4, 2, 64, 96)):
        # BASELINE config 4 (C=192, 6 heads): masked-out fraction 25 ... 100 %; the model configs: 0 and 50 %
        for drop in ((0.0, 0.25, 0.5, 0.75, 1.0) if heads == 6 else (0.0, 0.5)):
            cfg = dict(C=C, heads=heads, ws=ws, shift=s, B=16, H=H, W=W, drop=drop, masked=True, seed=5)
            p = G.attention_inputs(cfg)
            if drop == 0.0:
                p["alpha"] = torch.ones_like(p["alpha"])
            m = pkg.MaskedWinBasedAttention(C, heads, ws, s)
            with torch.no_grad():
                m.attn.qkv.weight.copy_(p["qkv_w"]); m.attn.qkv.bias.copy_(p["qkv_b"])
                m.attn.proj.weight.copy_(p["proj_w"]); m.attn.proj.bias.copy_(p["proj_b"])
                m.attn.relative_position_bias_table.copy_(p["table"])
            m = m.to(dev)
            x, a = p["x"].to(dev), p["alpha"].to(dev)
            kept = int(R.window_keep(p["alpha"], ws, s).sum())
            nwin = 16 * (H // ws) * (W // ws)
            flops = kept * R.flops_per_window(C, ws)
            byts = nwin * (2 * ws * ws * C * 4 + ws * ws * 4)
            res = {}
            algos = [("auto", pkg.ALGO_AUTO)]
            if not args.no_simt:
                algos.insert(0, ("simt", pkg.ALGO_SIMT))
            for name, algo in algos:
                m.algo = algo
                try:
                    with torch.no_grad():
                        y = m(x, a)
                        med, best = timeit(lambda: m(x, a), args.iters if name != "simt" else 2, flush)
                except pkg.MwaB200Error as e:
                    print(f"attn C={C} h={heads} ws={ws} drop={drop} {name}: {e}")
                    continue
                res[name] = y
                print(f"attn C={C} h={heads} ws={ws} s={s} kept {kept}/{nwin} {name:8s} median {med:8.3f} ms best {best:8.3f} "
                      f"{flops / med / 1e9:8.1f} TFLOP/s = {flops / med / 1e9 / PEAKS['bf16_tflops'] * 100:5.2f}% tensor peak; "
                      f"{byts / med / 1e6:7.1f} GB/s = {byts / med / 1e6 / PEAKS['hbm_gbs'] * 100:5.1f}% HBM", flush=True)
            if drop == 0.0:      # the alpha-free twin (layers/win_attention.py): every window kept, no residual copy pass
                mu = pkg.WinBasedAttention(C, heads, ws, s)
                mu.load_state_dict(m.state_dict())
                mu = mu.to(dev)
                with torch.no_grad():
                    yu = mu(x)
                    med, best = timeit(lambda: mu(x), args.iters, flush)
                print(f"attn C={C} h={heads} ws={ws} s={s} unmasked twin       auto     median {med:8.3f} ms best {best:8.3f} "
                      f"{flops / med / 1e9:8.1f} TFLOP/s = {flops / med / 1e9 / PEAKS['bf16_tflops'] * 100:5.2f}% tensor peak; "
                      f"max |unmasked - masked(alpha=1)| {(yu - res['auto']).abs().max().item():.1e}", flush=True)
            if "simt" in res and "auto" in res:
                d = (res["simt"] - res["auto"]).abs()
                print(f"    auto vs simt: max abs diff {d.max().item():.3e}, "
                      f"allclose(1e-3,1e-4) {torch.allclose(res['auto'], res['simt'], rtol=1e-3, atol=1e-4)}",
                      flush=True)


def bench_gate(args, dev, flush):
    a, b, x = (torch.randn(16, 192, 128, 192, device=dev) for _ in range(3))
    byts = a.numel() * 16
    with torch.no_grad():
        med, _ = timeit(lambda: pkg.gate_residual(a, b, x), args.iters, flush)
        print(f"gate_residual (16,192,128,192) fused kernel : median {med * 1e3:8.1f} us  {byts / med / 1e6:8.1f} GB/s = "
              f"{byts / med / 1e6 / PEAKS['hbm_gbs'] * 100:5.1f}% HBM", flush=True)
        med2, _ = timeit(lambda: a * torch.sigmoid(b) + x, args.iters, flush)
        print(f"    the reference's three torch kernels     : median {med2 * 1e3:8.1f} us  ({med2 / med:.2f}x)", flush=True)


def bench_round(args, dev, flush):
    y = torch.randn(16, 80, 64, 96, device=dev) * 4
    mu = torch.randn_like(y)
    big = torch.randn(64 * 1024 * 1024, device=dev)
    for name, fn, byts in (("quantize_offset y (16,80,64,96)", lambda: pkg.quantize_offset(y, mu), y.numel() * 12),
                           ("ste_round 256 MB", lambda: pkg.ste_round(big), big.numel() * 8)):
        med, best = timeit(fn, args.iters, flush)
        print(f"{name}: median {med * 1e3:8.1f} us  {byts / med / 1e6:8.1f} GB/s = "
              f"{byts / med / 1e6 / PEAKS['hbm_gbs'] * 100:5.1f}% HBM", flush=True)


def bench_pyramid(args, dev, flush):
    """alpha pyramid (+ mask quantisation) at the BASELINE config-2 shape vs the reference's op sequence in torch"""
    a = torch.rand(16, 1, 512, 768, device=dev)
    pool = torch.nn.AvgPool2d(3, stride=2, padding=1)

    def eager():
        r = torch.round(a * 255) / 255
        out, m = [], r
        for _ in range(6):
            m = pool(m)
            out.append(m)
        return r, out
    def graphed(fn, reps=10):
        """device time of one call: `reps` calls captured into one CUDA graph (these ops are shorter than the host
        takes to issue them, so event timing of eager calls would measure Python)"""
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            fn()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=s):
                for _ in range(reps):
                    keep = fn()
        med, best = timeit(gr.replay, args.iters, flush)
        return med / reps, best / reps
    med, best = graphed(lambda: pkg.alpha_pyramid(a, 6, quant_levels=255))
    med_e, best_e = graphed(eager)
    r0, l0 = pkg.alpha_pyramid(a, 6, quant_levels=255)
    r1, l1 = eager()
    r2 = torch.round(a.cpu() * 255) / 255
    l2, m = [], r2
    for _ in range(6):
        m = pool(m)
        l2.append(m)
    same_cpu = torch.equal(r0.cpu(), r2) and all(torch.equal(x.cpu(), y) for x, y in zip(l0, l2))
    diff_gpu = max((x - y).abs().max().item() for x, y in zip(l0, l1))
    nbytes = a.numel() * 4 * 2 + sum(x.numel() for x in l0) * 4
    print(f"alpha pyramid 16x1x512x768 (quantise + 6 levels), device time from a CUDA graph of 10 calls: 2 launches "
          f"{med * 1e3:6.1f} us ({nbytes / med / 1e6:6.0f} GB/s);  torch eager op sequence (9 launches) {med_e * 1e3:6.1f} us;  "
          f"bit-identical with torch CPU: {same_cpu};  max |diff| vs torch CUDA: {diff_gpu:.1e}")


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("what", nargs="*", default=["gdn", "attn", "round"])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--no-simt", action="store_true", help="skip the (slow) fp32 SIMT attention kernel")
    ap.add_argument("--lib", default=None, help="development: time a variant library (tools/build_variants.py)")
    args = ap.parse_args()
    if args.lib:
        pkg._abi.LIB_PATH = os.path.abspath(args.lib)
        print(f"variant library {args.lib}")
    dev = torch.device("cuda:0")
    flush = torch.zeros(128 * 1024 * 1024, device=dev)
    for w in args.what:
        {"gdn": bench_gdn, "attn": bench_attn, "round": bench_round, "gate": bench_gate, "pyramid": bench_pyramid}[w](args, dev, flush)
