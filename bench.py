#!/usr/bin/env python
"""Benchmark on B200: the RGBA codec's encode + decode forward, its hot path, and the kernels' rooflines.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--legs forward,hotpath,config4,config5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload "C2-forward" (BASELINE.json configs[1], per GPU): the full AutoEncoderRGB_Journal encode + decode forward
(<package>/codec.py: the reference's module tree on the B200 modules, convolutions on the tcgen05 kernel) on a batch of
16 synthetic 768x512 RGBA images, random-init weights.  A "step" is one forward of the batch incl. the alpha pyramids.
value = images/s = 16 * N / step time (device time, max over ranks); e2e = the same with the RGBA batch coming from
pinned host memory and x_hat going back, copies inside the timed region.  Images are independent -> ranks shard by image
with no collective (weak scaling, 16 images per GPU).  The hot-path kernels are timed live inside the same steps with
CUDA events around the module calls; `roofline` is the masked window-attention kernel the metric names.
Extra legs on the same JSON line: `hotpath` (round 1's workload: only the hot-path call sites, back to back),
`config4` (attention microbench, 6 heads, 0-100 % masked), `config5` (training step of the codec on 256x256 crops with
the NCCL gradient all-reduce).  Prints ONE JSON line (rank 0).
--dump-outputs DIR writes what the last timed forward step returned (rank 0's shard) as DIR/<name>.npy, so that two
builds run with the same arguments (same seeded inputs and weights) can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "768x512 RGBA images/s (AutoEncoderRGB_Journal encode + decode forward); masked-attn kernel % of roofline"
UNIT = "images/s"
BATCH_PER_GPU = 16
IMG_H, IMG_W = 512, 768
ATTN_SITES = [  # name, C, heads, ws, shift, scale divisor, which pyramid level feeds alpha
    ("enc.attention1", 192, 8, 8, 4, 4, 1), ("enc.attention2", 80, 8, 4, 2, 8, 2),
    ("dec.attention1", 80, 8, 4, 2, 8, 2), ("dec.attention2", 192, 8, 8, 4, 4, 1)]
GDN_SITES = [("enc.gdn1", 2, False), ("enc.gdn2", 4, False), ("enc.gdn3", 8, False),
             ("dec.igdn1", 8, True), ("dec.igdn2", 4, True), ("dec.igdn3", 2, True)]
FLOPS_PER_WINDOW = {(192, 8): 8 * 64 * 192 * 192 + 4 * 64 * 64 * 192, (80, 4): 8 * 16 * 80 * 80 + 4 * 16 * 16 * 80}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm=float(p["hbm_gbs"]), tensor=float(p["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, tensor=1590.0, source="fallback")


# ------------------------------------------------------------------------------------------------ inputs
def synthetic_alpha(batch: int, seed0: int) -> torch.Tensor:
    """union of seeded ellipses (~50 % coverage), 3-px linear soft edge, values k/255  (SURVEY.md 8d, C1/C2)"""
    ys = torch.arange(IMG_H, dtype=torch.float32)[:, None]
    xs = torch.arange(IMG_W, dtype=torch.float32)[None, :]
    out = torch.zeros(batch, 1, IMG_H, IMG_W)
    for b in range(batch):
        g = torch.Generator().manual_seed(seed0 + b)
        d = torch.full((IMG_H, IMG_W), -1e9)
        for _ in range(4):
            cy, cx = torch.rand(2, generator=g).tolist()
            ry, rx = (0.15 + 0.2 * torch.rand(2, generator=g)).tolist()
            r = torch.sqrt(((ys - cy * IMG_H) / (ry * IMG_H)) ** 2 + ((xs - cx * IMG_W) / (rx * IMG_W)) ** 2)
            d = torch.maximum(d, (1.0 - r) * min(ry * IMG_H, rx * IMG_W))      # ~signed distance in px
        out[b, 0] = torch.round(torch.clamp(d / 3.0, 0.0, 1.0) * 255) / 255
    return out


def _host_pyramid(alpha: torch.Tensor, levels: int = 6):
    """me1..me6 of the synthetic alpha (plain torch on the host: input generation, layers/SupplyMask.py:10-18)"""
    out, a = [], alpha
    for _ in range(levels):
        a = torch.nn.functional.avg_pool2d(a, 3, stride=2, padding=1)
        out.append(a)
    return out


def _host_kept_windows(alpha: torch.Tensor, ws: int, s: int) -> torch.Tensor:
    """bool (B * nW,): which windows of the cyclically shifted alpha are not all-zero (bookkeeping for the FLOP count)"""
    B, _, H, W = alpha.shape
    a = torch.roll(alpha[:, 0], shifts=(-s, -s), dims=(1, 2)) if s > 0 else alpha[:, 0]
    return (a.reshape(B, H // ws, ws, W // ws, ws) != 0).any(dim=4).any(dim=2).reshape(-1)


def build_workload(pkg, dev, batch: int, seed0: int):
    """modules with random-init weights (torch.manual_seed(234), the scripts' default) + synthetic inputs"""
    torch.manual_seed(234)
    alpha = synthetic_alpha(batch, seed0)
    pyr = _host_pyramid(alpha)                        # me1..me6 (CPU, input generation only)
    gen = torch.Generator().manual_seed(seed0 + 999)
    ops = []
    for name, C, heads, ws, shift, div, lvl in ATTN_SITES:
        m = pkg.MaskedWinBasedAttention(C, heads, ws, shift)
        with torch.no_grad():
            m.attn.relative_position_bias_table.normal_(0, 0.02, generator=gen)
        x = torch.randn(batch, C, IMG_H // div, IMG_W // div, generator=gen)
        a = pyr[lvl].contiguous()
        keep = _host_kept_windows(a, ws, shift)
        ops.append(dict(kind="attn", name=name, mod=m.to(dev), x=x, alpha=a, kept=int(keep.sum()),
                        windows=int(keep.numel()), C=C, ws=ws, heads=heads, shift=shift))
    for name, div, inverse in GDN_SITES:
        m = pkg.GDN(192, inverse=inverse)
        with torch.no_grad():
            m.gamma.add_(torch.rand(192, 192, generator=gen) * 0.02)
            m.beta.mul_(0.5 + torch.rand(192, generator=gen))
        x = torch.randn(batch, 192, IMG_H // div, IMG_W // div, generator=gen)
        ops.append(dict(kind="gdn", name=name, mod=m.to(dev), x=x, inverse=inverse))
    y = torch.randn(batch, 80, IMG_H // 8, IMG_W // 8, generator=gen) * 4
    mu = torch.randn(batch, 80, IMG_H // 8, IMG_W // 8, generator=gen)
    lrp = torch.randn(batch, 80, IMG_H // 8, IMG_W // 8, generator=gen)
    z = torch.randn(batch, 192, IMG_H // 64, IMG_W // 64, generator=gen) * 3
    med = torch.randn(1, 192, 1, 1, generator=gen) * 0.1
    ops.append(dict(kind="round", name="latent rounding (reconmask, z, 10 y slices + lrp)", y=y, mu=mu, lrp=lrp, z=z,
                    med=med, mask=alpha))
    return ops


def to_device(ops, dev, pin=False):
    for op in ops:
        for k, v in list(op.items()):
            if isinstance(v, torch.Tensor):
                if pin:
                    op["h_" + k] = v.pin_memory()
                op[k] = v.to(dev)
    return ops


def run_op(pkg, op, t=None):
    """one hot-path call site; t overrides the device inputs (used by the e2e leg). returns list of outputs"""
    g = (lambda k: t[k]) if t is not None else (lambda k: op[k])
    if op["kind"] == "attn":
        return [op["mod"](g("x"), g("alpha"))]
    if op["kind"] == "gdn":
        return [op["mod"](g("x"))]
    outs = [pkg.quantize_levels(g("mask"), 255), pkg.quantize_offset(g("z"), g("med"))]
    ys, mus, lrps = g("y").chunk(10, 1), g("mu").chunk(10, 1), g("lrp").chunk(10, 1)
    for i in range(10):
        yh = pkg.quantize_offset(ys[i], mus[i])
        outs.append(pkg.lrp_add(yh, lrps[i]))
    return outs


# our kernels per step: 4 attention calls x (scan, compact, residual copy, main) + 6 GDN + 22 rounding
LAUNCHES_PER_STEP = 4 * 4 + 6 + (2 + 20)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        rows = [r for ts, r in self.rows if t0 - 0.05 <= ts <= t1 + 0.15] or [r for _, r in self.rows]
        for r in rows:
            f = [c.strip() for c in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}




# ------------------------------------------------------------------------------------------------ plumbing
def _env():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0")))


class Dist:
    """barrier + max-over-ranks on the device (NCCL); the inference data path has no collective"""

    def __init__(self, dev, world):
        self.dev, self.world, self.dist = dev, world, None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=dev)
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_ms(self, ms: float) -> float:
        t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def timed_steps(fn, steps, warmup, D: Dist):
    """W untimed steps, then exactly K steps between barrier + synchronize, CUDA events on the launching stream"""
    for _ in range(warmup):
        fn()
    D.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    D.barrier()
    return D.max_ms(e0.elapsed_time(e1)) / steps, t0, time.time()


# AutoEncoder.forward's return values (<package>/codec.py), in order
FORWARD_OUTPUTS = ("x_hat", "mse", "bpp", "bpp_y", "bpp_z")
DUMP_SAMPLE = 1 << 23            # elements kept of a larger output: 32 MB in float32, the whole dump stays under 64 MB
DUMP_SEED = 0


def dump_outputs(out_dir: str, names, tensors) -> None:
    """DIR/<name>.npy per output, float64 kept, anything else as float32.  An output of more than DUMP_SAMPLE elements
    is stored as flat[idx] with idx = sorted(randperm(numel, seed DUMP_SEED)[:DUMP_SAMPLE]): the same elements on every
    run with the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in zip(names, tensors, strict=True):
        t = t.detach()
        t = t if t.dtype == torch.float64 else t.float()
        flat = t.reshape(-1)
        if flat.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(DUMP_SEED)
            idx = torch.randperm(flat.numel(), generator=g)[:DUMP_SAMPLE].sort().values
            arr = flat[idx.to(flat.device)].cpu().numpy()
        else:
            arr = t.cpu().numpy()
        total += arr.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    assert total <= 64 << 20, total


# ------------------------------------------------------------------------------------------------ the codec workload
def synthetic_rgba(batch: int, seed0: int) -> torch.Tensor:
    """(B, 4, H, W) in [0, 1]: smooth colour fields + noise, alpha = soft ellipse blobs; the colour planes are zero
    where alpha is (what the dataset feeds: my_datasets pre-multiply by the binarised alpha)"""
    alpha = synthetic_alpha(batch, seed0)
    yy = torch.linspace(0, 1, IMG_H).view(1, 1, IMG_H, 1)
    xx = torch.linspace(0, 1, IMG_W).view(1, 1, 1, IMG_W)
    out = torch.empty(batch, 4, IMG_H, IMG_W)
    for b in range(batch):
        g = torch.Generator().manual_seed(seed0 + b + 5000)
        f = (1.0 + 4.0 * torch.rand(6, generator=g)).tolist()
        rgb = torch.cat([0.5 + 0.4 * torch.sin(6.28 * (f[0] * xx + f[1] * yy)), 0.5 + 0.4 * torch.cos(6.28 * (f[2] * yy - f[3] * xx)),
                         0.5 + 0.3 * torch.sin(6.28 * (f[4] * xx * yy) + f[5])], dim=1)[0]
        rgb = (rgb + 0.05 * torch.randn(3, IMG_H, IMG_W, generator=g)).clamp(0, 1)
        out[b, :3] = rgb * (alpha[b] > 0).float()
        out[b, 3] = alpha[b, 0]
    return out


class OpTimer:
    """CUDA events around every hot-path module call (forward hooks), recorded on the launching stream inside the timed
    steps: the per-kernel durations behind `rooflines` are measured live, in the run that prints them"""

    def __init__(self, net, pkg):
        self.names, self.events, self.on = [], {}, False
        for name, m in net.named_modules():
            if isinstance(m, (pkg.GDN, pkg.MaskedWinBasedAttention)):
                self.names.append(name)
                self.events[name] = []
                m.register_forward_pre_hook(self._pre(name))
                m.register_forward_hook(self._post(name))

    def _pre(self, name):
        def hook(mod, args):
            if self.on:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                self.events[name].append([e, None])
        return hook

    def _post(self, name):
        def hook(mod, args, out):
            if self.on:
                e = torch.cuda.Event(enable_timing=True)
                e.record()
                self.events[name][-1][1] = e
        return hook

    def mean_ms(self):
        return {n: statistics.mean(a.elapsed_time(b) for a, b in ev) for n, ev in self.events.items() if ev}


# hot-path kernels per forward: 2 alpha pyramids (2 + 1 launches), 4 attention calls x (scan, compact, dropped-window copy,
# main), 6 GDN, z rounding; the gate, the slice quantisation and the lrp update are convolution epilogues.  The
# convolution launches (kernel + plane-split launches) are counted live by the binding (_abi.launch_count).
LAUNCHES_PER_FORWARD = 3 + 4 * 4 + 6 + 1
# round 1's hot-path-only step: 4 attention calls x 4 + 6 GDN + 22 rounding launches
LAUNCHES_PER_HOTPATH_STEP = 4 * 4 + 6 + (2 + 20)


def traffic_table():
    """DRAM bytes per launch from the committed `ncu --set full` captures (tools/ncu_traffic.py writes the table together
    with the sha256 of the capture it was read from and the digest of the library that was profiled)"""
    path = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(path):
        return {}
    with open(path) as f:
        return json.load(f)


def leg_forward(pkg, dev, rank, world, D, args, pk, tf32_convs=False, steps=None, want_e2e=True, sampler=None, library_convs=False,
                dump_dir=None):
    pkg.conv.USE_KERNEL = not library_convs
    torch.backends.cudnn.allow_tf32 = bool(tf32_convs)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(234)
    net = pkg.RGBACodec().eval().to(dev)
    timer = OpTimer(net, pkg)
    rgba_host = synthetic_rgba(BATCH_PER_GPU, seed0=BATCH_PER_GPU * rank).pin_memory()
    rgba = rgba_host.to(dev)
    image, alpha = rgba[:, :3].contiguous(), rgba[:, 3:4].contiguous()

    last = {}

    def step(img=image, a=alpha):
        me = net.EncMakeMask(a)                                  # trainRGB.py:283
        last["out"] = net(img, a, a, me[0], me[1], me[2], me[3])     # trainRGB.py:289 (reconmask = the alpha itself)
        return last["out"]

    steps = steps or args.steps
    with torch.no_grad():
        for _ in range(args.warmup):
            step()
        D.barrier()
        if sampler is not None:                                  # keep the GPU under load until the sampler is live
            t_dead = time.time() + 4.0
            while not sampler.rows and time.time() < t_dead and sampler.proc is not None:
                step()
                torch.cuda.synchronize()
        n0 = pkg._abi.launch_count
        step()
        conv_launches = pkg._abi.launch_count - n0               # convolution kernels + plane splits + rate terms of one forward
        timer.on = True
        ms_per_step, t0, t1 = timed_steps(step, steps, 0, D)
        timer.on = False
        if dump_dir is not None and rank == 0:
            dump_outputs(dump_dir, FORWARD_OUTPUTS, last["out"])
    clocks = sampler.stop(t0, t1) if sampler is not None else None
    per_op = timer.mean_ms()
    value = BATCH_PER_GPU * world / (ms_per_step * 1e-3)

    # ---- rooflines of the hot-path kernels inside the forward (rank 0's kernels): algorithmic work / measured duration
    pyr = _host_pyramid(rgba_host[:, 3:4])
    traffic = traffic_table()
    roofs = []
    big = [n for n in per_op if n.endswith("attention1.attn") and n.startswith("Encoder") or
           n.endswith("attention2.attn") and n.startswith("Decoder")]
    kept8 = int(_host_kept_windows(pyr[1].contiguous(), 8, 4).sum())
    nwin8 = BATCH_PER_GPU * (IMG_H // 32) * (IMG_W // 32)
    if big:
        ms8 = sum(per_op[n] for n in big)
        fl8 = len(big) * kept8 * FLOPS_PER_WINDOW[(192, 8)]
        t8 = traffic.get("attention_8x8")
        roofs.append({"kernel": "masked window attention 8x8 C=192, split-precision tcgen05 (op = scan + compact + dropped-window "
                                f"copy + main kernel; {len(big)} ops/step)",
                      "bound": "tensor", "achieved": fl8 / (ms8 * 1e-3) / 1e12, "peak": pk["tensor"], "unit": "TFLOP/s",
                      "frac": fl8 / (ms8 * 1e-3) / 1e12 / pk["tensor"],
                      "traffic": t8["dram_bytes_per_launch"] if t8 else None, "traffic_source": t8["source"] if t8 else None,
                      "hbm_gbs": len(big) * nwin8 * 98560 / (ms8 * 1e-3) / 1e9, "ms_per_op": ms8 / len(big),
                      "kept_windows_per_op": kept8, "windows_per_op": nwin8,
                      "note": "algorithmic FLOPs (22.02 MFLOP per kept window) over the bf16 dense peak; the kernel runs "
                              "3 fp16 passes per contraction to be fp32-faithful, so its own ceiling is peak / 3"})
    small = [n for n in per_op if n.endswith(".attn") and n not in big]
    if small:
        kept4 = int(_host_kept_windows(pyr[2].contiguous(), 4, 2).sum())
        ms4 = sum(per_op[n] for n in small)
        by4 = len(small) * BATCH_PER_GPU * (IMG_H // 32) * (IMG_W // 32) * 10304
        roofs.append({"kernel": f"masked window attention 4x4 C=80, fp32 ({len(small)} ops/step)", "bound": "hbm",
                      "achieved": by4 / (ms4 * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                      "frac": by4 / (ms4 * 1e-3) / 1e9 / pk["hbm"], "traffic": None, "ms_per_op": ms4 / len(small),
                      "tflops": len(small) * kept4 * FLOPS_PER_WINDOW[(80, 4)] / (ms4 * 1e-3) / 1e12})
    gdn = [n for n in per_op if "gdn" in n]
    if gdn:
        px = BATCH_PER_GPU * sum((IMG_H // d) * (IMG_W // d) for d in (2, 4, 8)) * 2
        msg = sum(per_op[n] for n in gdn)
        tg = traffic.get("gdn")
        roofs.append({"kernel": f"GDN/IGDN C=192 ({len(gdn)} launches/step)", "bound": "hbm",
                      "achieved": px * 1536 / (msg * 1e-3) / 1e9, "peak": pk["hbm"], "unit": "GB/s",
                      "frac": px * 1536 / (msg * 1e-3) / 1e9 / pk["hbm"],
                      "traffic": tg["dram_bytes_per_step"] if tg else None, "traffic_source": tg["source"] if tg else None,
                      "ms_per_step": msg,
                      "note": "1536 B per pixel (fp32 in, 4 B per element out); gdn1 / gdn3 / igdn1 / igdn3 write the fp16 hi / lo "
                              "planes their consumer convolution reads (gdn_forward_planes: same bytes, no fp32 tensor and no "
                              "split launch behind them), gdn2 / igdn2 the dense tensor the attention reads"})
    hot_ms = sum(per_op.values())

    # ---- e2e: RGBA batch from pinned host memory -> H2D -> forward -> x_hat D2H, all inside the timed region
    e2e = None
    if want_e2e:
        n = max(4, min(steps, 8))
        out_hosts = [torch.empty(BATCH_PER_GPU, 3, IMG_H, IMG_W).pin_memory() for _ in range(2)]
        pipe = pkg.HostPipeline(net, dev)

        def e2e_run():           # n steps through the package's host pipeline: every step's batch comes from pinned host
            pipe.run([rgba_host] * n, [out_hosts[i & 1] for i in range(n)])     # memory and its x_hat goes back to it

        with torch.no_grad():
            e2e_run()
            ms_all, _, _ = timed_steps(e2e_run, 1, 0, D)
        ms_e2e = ms_all / n
        e2e = {"value": BATCH_PER_GPU * world / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": rgba_host.numel() * 4,
               "d2h_bytes_per_step": out_hosts[0].numel() * 4, "ms_per_step": ms_e2e, "steps": n,
               "how": "HostPipeline.run: every step's pinned host RGBA batch -> H2D -> AutoEncoder.forward (alpha pyramids, "
                      "analysis, hyperprior, slice loop, synthesis, bpp) -> D2H of x_hat into pinned host memory; all copies "
                      "inside the timed region, on two copy streams that overlap the neighbouring steps' compute (two "
                      "staging slots); time = whole run of n steps incl. pipeline fill and drain, / n"}
    del net
    torch.cuda.empty_cache()
    return dict(value=value, ms_per_step=ms_per_step, per_op_ms=per_op, rooflines=roofs, e2e=e2e, clocks=clocks,
                hot_path_ms_per_step=hot_ms, hot_path_share=hot_ms / ms_per_step, steps=steps, conv_launches=conv_launches)


# ------------------------------------------------------------------------------------------------ hot path only
def leg_hotpath(pkg, dev, rank, world, D, args, pk, steps):
    """round 1's workload: the hot-path call sites of one forward, back to back, inputs resident (13.9 GB per step)"""
    ops = to_device(build_workload(pkg, dev, BATCH_PER_GPU, seed0=BATCH_PER_GPU * rank), dev)
    stream = torch.cuda.current_stream()
    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            for op in ops:
                run_op(pkg, op)
        D.barrier()
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(len(ops) + 1)] for _ in range(steps)]
        for s in range(steps):
            ev[s][0].record(stream)
            for i, op in enumerate(ops):
                run_op(pkg, op)
                ev[s][i + 1].record(stream)
        D.barrier()
    ms = D.max_ms(ev[0][0].elapsed_time(ev[-1][-1])) / steps
    per_op = [statistics.mean(ev[s][i].elapsed_time(ev[s][i + 1]) for s in range(steps)) for i in range(len(ops))]
    big = [(op, t) for op, t in zip(ops, per_op) if op["kind"] == "attn" and op["C"] == 192]
    fl = sum(op["kept"] * FLOPS_PER_WINDOW[(192, 8)] for op, _ in big)
    tb = sum(t for _, t in big)
    gd = [(op, t) for op, t in zip(ops, per_op) if op["kind"] == "gdn"]
    gb = sum(op["x"].numel() // 192 * 1536 for op, _ in gd)
    tg = sum(t for _, t in gd)
    rnd_ms = sum(t for op, t in zip(ops, per_op) if op["kind"] == "round")
    rnd_bytes = BATCH_PER_GPU * (491520 * (12 + 12) + 18432 * 8 + IMG_H * IMG_W * 8)
    res = {"value": BATCH_PER_GPU * world / (ms * 1e-3), "unit": "images/s (hot-path call sites only)", "ms_per_step": ms,
           "steps": steps, "gpu_launches": LAUNCHES_PER_HOTPATH_STEP * steps,
           "per_op_ms": {op["name"]: t for op, t in zip(ops, per_op)},
           "attention_8x8": {"tflops": fl / (tb * 1e-3) / 1e12, "frac_of_tensor_peak": fl / (tb * 1e-3) / 1e12 / pk["tensor"],
                             "kept": f'{big[0][0]["kept"]}/{big[0][0]["windows"]}', "ms_per_op": tb / len(big)},
           "gdn": {"gbs": gb / (tg * 1e-3) / 1e9, "frac_of_hbm_peak": gb / (tg * 1e-3) / 1e9 / pk["hbm"], "ms_per_step": tg},
           "rounding": {"gbs": rnd_bytes / (rnd_ms * 1e-3) / 1e9, "frac_of_hbm_peak": rnd_bytes / (rnd_ms * 1e-3) / 1e9 / pk["hbm"],
                        "ms_per_step": rnd_ms}}
    del ops
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ BASELINE config 4
def leg_config4(pkg, dev, pk, iters=8):
    """masked window-attention microbench: 8x8 windows, C = 192, 6 heads, 0 / 25 / 50 / 75 / 100 % of the windows masked
    out, as blobs (4 x 4 windows, what transparent regions of real images look like) and as independent windows (the
    worst case for the gather: no neighbour shares a sector).  L2 flushed between launches."""
    flush = torch.zeros(128 * 1024 * 1024, device=dev)
    torch.manual_seed(3)
    m = pkg.MaskedWinBasedAttention(192, 6, 8, 4).to(dev)
    x = torch.randn(16, 192, 128, 192, device=dev)
    out = {}
    with torch.no_grad():
        for pattern, cell in (("blobs", 4), ("independent", 1)):
            rows = {}
            for masked in (0.0, 0.25, 0.5, 0.75, 1.0):
                g = torch.Generator(device=dev).manual_seed(int(masked * 100) + cell)
                keep = (torch.rand(16, 1, 16 // cell, 24 // cell, device=dev, generator=g) >= masked).float()
                a = torch.roll(keep.repeat_interleave(8 * cell, 2).repeat_interleave(8 * cell, 3), (4, 4), (2, 3))
                kept = int(keep.sum().item()) * cell * cell
                for _ in range(2):
                    m(x, a)
                ts = []
                for _ in range(iters):
                    flush.add_(1.0)
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); m(x, a); e1.record(); torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1))
                ms = statistics.median(ts)
                tf = kept * FLOPS_PER_WINDOW[(192, 8)] / (ms * 1e-3) / 1e12
                rows[f"{int(masked * 100)}%"] = {"ms": ms, "kept_windows": kept, "tflops": tf, "frac_of_tensor_peak": tf / pk["tensor"],
                                                 "hbm_gbs": 6144 * 98560 / (ms * 1e-3) / 1e9}
            out[pattern] = rows
    del flush
    torch.cuda.empty_cache()
    return {"workload": "C4: MaskedWinBasedAttention(192, 6 heads, ws 8, shift 4) on (16, 192, 128, 192) = 6144 windows, "
                        "default (fp32-faithful) kernel, median of %d launches, L2 flushed" % iters, "masked_out": out}


# ------------------------------------------------------------------------------------------------ BASELINE config 5
def leg_config5(pkg, dev, rank, world, D, steps=6, warmup=2):
    """RGBA training step on 256x256 crops, 8 per GPU (batch 64 on 8 GPUs): forward + backward of the whole codec (our
    backward kernels under the drop-in modules, cuDNN for the convolutions), rate-distortion loss as trainRGB.py:176-186,
    bucketed NCCL gradient all-reduce + the reference's +-5 clip after the reduction, Adam step."""
    crop, per_gpu = 256, 8
    torch.backends.cudnn.allow_tf32 = False
    torch.manual_seed(234)
    net = pkg.RGBACodec().train().to(dev)
    params = [p for p in net.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=1e-4)
    ar = pkg.GradientAllReduce(params, clip_value=5.0)
    g = torch.Generator().manual_seed(1000 + rank)
    img = torch.rand(per_gpu, 3, crop, crop, generator=g).to(dev)
    a = (torch.rand(per_gpu, 1, crop // 32, crop // 32, generator=g) > 0.35).float().repeat_interleave(32, 2).repeat_interleave(32, 3).to(dev)
    img = img * a
    ms_parts = {}

    def fwd_bwd():
        me = net.EncMakeMask(a)
        x_hat, mse, bpp, _, _ = net(img, a, a, me[0], me[1], me[2], me[3])
        loss = 4096 * mse + bpp
        opt.zero_grad(set_to_none=True)
        loss.backward()

    def step():
        fwd_bwd()
        ar()
        opt.step()

    ms, _, _ = timed_steps(step, steps, warmup, D)
    ms_fb, _, _ = timed_steps(fwd_bwd, max(2, steps // 2), 0, D)
    ms_ar, _, _ = timed_steps(ar, max(2, steps // 2), 0, D)
    nparam = sum(p.numel() for p in params)
    res = {"workload": "C5: AutoEncoderRGB_Journal training step, 256x256 crops, 8 per GPU, fwd + bwd + bucketed gradient "
                       "all-reduce (NCCL) + clip + Adam", "value": per_gpu * world / (ms * 1e-3), "unit": "crops/s",
           "ms_per_step": ms, "fwd_bwd_ms": ms_fb, "grad_exchange_ms": ms_ar, "grad_bytes": 4 * nparam, "global_batch": per_gpu * world,
           "steps": steps, "weight_gradient_gemms": "fp32" if not pkg._abi.WGRAD_TF32 else "tf32 products (opt-in)"}
    if world > 1:
        res["allreduce_busbw_gbs"] = 2 * (world - 1) / world * 4 * nparam / (ms_ar * 1e-3) / 1e9
    del net, opt, ar
    torch.cuda.empty_cache()
    return res


# ------------------------------------------------------------------------------------------------ CPU legs
def cpu_forward_images_per_s(seconds_budget: float, max_passes: int = 200):
    """the oracle port (oracle/ref_model.py = the reference's AutoEncoder.forward restated on torch CPU, pinned on outputs
    of the unmodified reference model; all host threads) on ONE synthetic 768x512 RGBA image per pass"""
    from oracle import golden_cases as G
    from oracle import ref_model as M
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    with open(os.path.join(ROOT, "tests", "golden", "model_rgb_keys.json")) as f:
        table = json.load(f)
    w = G.model_state(table, 234)
    rgba = synthetic_rgba(1, seed0=0)
    image, alpha = rgba[:, :3].contiguous(), rgba[:, 3:4].contiguous()
    with torch.no_grad():
        M.rgb_forward(w, image, alpha, alpha)             # warm-up
        times = []
        t_start = time.perf_counter()
        while len(times) < 3 or (time.perf_counter() - t_start < seconds_budget and len(times) < max_passes):
            t0 = time.perf_counter()
            M.rgb_forward(w, image, alpha, alpha)
            times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    sample = (f"{len(times)} passes of the full encode + decode forward on 1 synthetic 768x512 RGBA image "
              f"(oracle/ref_model.py), torch CPU fp32, {cores} threads, median")
    return 1.0 / med, cores, sample, med


def cpu_config1_hot_path_ms():
    """BASELINE config 1: AutoEncoderMask_Journal on one 768x512 alpha mask on CPU -- its hot path is the six GDN / IGDN
    of models/AutoEncoderMask_Journal.py:153-176 (192 channels at 1/2, 1/4, 1/8 scale); oracle port, all host threads"""
    from oracle import ref_ops as R
    gen = torch.Generator().manual_seed(1)
    pedestal = 2.0 ** -36
    beta = torch.sqrt(torch.ones(192) + pedestal)
    gamma = torch.sqrt(0.1 * torch.eye(192) + torch.rand(192, 192, generator=gen) * 0.01 + pedestal)
    xs = [torch.randn(1, 192, IMG_H // d, IMG_W // d, generator=gen) for d in (2, 4, 8, 8, 4, 2)]
    def one():
        for i, x in enumerate(xs):
            R.gdn(x, beta, gamma, inverse=i >= 3)
    with torch.no_grad():
        one()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); one(); ts.append(time.perf_counter() - t0)
    return statistics.median(ts) * 1e3


def reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference is pure Python and cannot travel
    to the GPU box, so this is the oracle port (kind 'port'), all host threads; every step is ONE image (a bounded sample
    of the batch-16 workload), at most K steps or ~150 s."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ips, cores, sample, med = cpu_forward_images_per_s(150.0, max_passes=max(args.steps, 3))
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "C2-forward: AutoEncoderRGB_Journal encode + decode forward, 768x512 RGBA, 1 image per CPU pass "
                               "(bounded sample of the batch-16 workload)"},
        "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--legs", default="forward,tf32,hotpath,config4,config5,config1",
                    help="comma list of the extra legs to run next to the headline forward")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="skip the nvidia-smi clock sampler (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed forward step as DIR/<name>.npy (a fixed, seeded sample of "
                         "x_hat; rank 0's shard)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU forward (--impl ours)")
    if args.impl == "reference":
        return reference_arm(args)
    args.warmup = max(args.warmup, 3)
    legs = set(args.legs.split(","))

    import mwa_b200 as pkg
    rank, world, local = _env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    D = Dist(dev, world)
    pk = peaks()

    sampler = ClockSampler(local) if (rank == 0 and not args.no_clocks) else None      # needs ~0.5 s to start
    fwd = leg_forward(pkg, dev, rank, world, D, args, pk, tf32_convs=False, want_e2e=not args.no_e2e, sampler=sampler,
                      dump_dir=args.dump_outputs)
    extra = {}
    if "tf32" in legs:
        for key, tf32 in (("forward_library_convs_fp32", False), ("forward_library_convs_tf32", True)):
            t = leg_forward(pkg, dev, rank, world, D, args, pk, tf32_convs=tf32, steps=max(3, min(args.steps, 5)), want_e2e=False,
                            library_convs=True)
            extra[key] = {"value": t["value"], "unit": UNIT, "ms_per_step": t["ms_per_step"], "steps": t["steps"],
                          "note": "same forward with every convolution through torch.nn.functional (cuDNN, "
                                  + ("allow_tf32 = True: torch's default, what the unmodified reference runs on a GPU"
                                     if tf32 else "fp32, TF32 off: the reference's arithmetic") + "); the hot-path kernels unchanged"}
        pkg.conv.USE_KERNEL = True
    if "hotpath" in legs:
        extra["hotpath"] = leg_hotpath(pkg, dev, rank, world, D, args, pk, steps=max(5, min(args.steps, 50)))
    if "config5" in legs:
        try:
            extra["config5_training"] = leg_config5(pkg, dev, rank, world, D)
        except Exception as exc:      # noqa: BLE001 -- an extra leg must not take the headline down
            extra["config5_training"] = {"error": repr(exc)[:300]}
    if "config4" in legs and rank == 0 and world == 1:
        extra["config4_attention_microbench"] = leg_config4(pkg, dev, pk)
    if "config1" in legs and rank == 0 and world == 1:
        torch.manual_seed(1)
        gd = [pkg.GDN(192, inverse=i >= 3).to(dev) for i in range(6)]
        xs = [torch.randn(1, 192, IMG_H // d, IMG_W // d, device=dev) for d in (2, 4, 8, 8, 4, 2)]
        with torch.no_grad():
            ms1, _, _ = timed_steps(lambda: [m(x) for m, x in zip(gd, xs)], 20, 3, D)
        extra["config1_mask_model_hot_path"] = {"workload": "C1: the six GDN / IGDN of AutoEncoderMask_Journal on one 768x512 "
                                                            "alpha mask (batch 1)", "gpu_ms": ms1}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ips, cores, sample, med = cpu_forward_images_per_s(12.0)
        cpu = {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
               "config1_hot_path_ms": cpu_config1_hot_path_ms()}

    if rank == 0:
        roofs = fwd["rooflines"]
        roofline = None
        if roofs:
            r0 = roofs[0]
            roofline = {k: r0.get(k) for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic", "traffic_source")}
            roofline["peak_source"] = (pk["source"] + " (MEASURED_PEAKS.json burst figures)") if pk["source"] == "measured" \
                else "fallback (B200_PROFILING.md)"
        gdn_r = next((r for r in roofs if r["kernel"].startswith("GDN")), None)
        per_forward = LAUNCHES_PER_FORWARD + fwd["conv_launches"]
        hot_launches = per_forward * fwd["steps"]
        line = {
            "metric": METRIC, "value": fwd["value"], "unit": UNIT, "n_gpus": world, "steps": fwd["steps"],
            "warmup": args.warmup, "ms_per_step": fwd["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f32 (attention: fp16 hi+lo split operands, 3 tcgen05 passes, f32 accumulate = f32-faithful; 4x4 attention "
                     "plain f32; GDN contraction bf16x3 split + f32 accumulate; convolutions fp16 hi+lo split operands, 3 tcgen05 passes, "
                     "chunked f32 accumulation outside the tensor core = f32-faithful)",
            "data": "synthetic",
            "config": {"workload": "C2-forward: AutoEncoderRGB_Journal encode + decode forward (alpha pyramids, analysis, "
                                   "hyperprior, 10-slice loop, synthesis, bpp), batch 16 x 768x512 RGBA per GPU, random-init "
                                   "weights (seed 234), alpha = soft ellipse blobs",
                       "images_per_gpu": BATCH_PER_GPU,
                       "l2": "activations of one step >> 126 MB L2 (1.2 GB per 1/2-scale tensor): inputs larger than L2, no flush",
                       "hot_path_share_of_step": fwd["hot_path_share"]},
            "roofline": roofline, "roofline_gdn": gdn_r, "rooflines": roofs, "cpu_baseline": cpu, "e2e": fwd["e2e"],
            "gpu_launches": hot_launches,
            "gpu_launches_note": f"{per_forward} launches of this repo's kernels per forward: {LAUNCHES_PER_FORWARD} hot-path launches "
                                 f"(alpha pyramids, attention, GDN, z rounding) + {fwd['conv_launches']} convolution / plane-split / "
                                 "rate-term launches counted by the binding (the masked squared error and the bpp terms are "
                                 "rate_forward's four launches)",
            "clocks": fwd["clocks"], "per_op_ms": fwd["per_op_ms"], "hot_path_ms_per_step": fwd["hot_path_ms_per_step"],
        }
        line.update(extra)
        print(json.dumps(line), flush=True)
    D.close()


if __name__ == "__main__":
    main()
