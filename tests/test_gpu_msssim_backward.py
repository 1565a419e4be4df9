"""Masked MS-SSIM as a training loss: the gradient of `masked_ms_ssim` (csrc/msssim.cu, ms_ssim_level_backward) against
fp64 autograd through the CPU oracle (oracle/ref_model.masked_ms_ssim), its exact properties, its launches and
synchronisations, the C ABI's argument checks, and one training step of the codec with it as the distortion term."""
import ctypes
import os
import warnings

import pytest
import torch

import bench
from oracle import golden_cases as G
from oracle import ref_model as M

gpu = pytest.mark.gpu

# Per element |grad - ref| <= REL * max|ref|.  fp32 autograd through the oracle on the CPU reaches ~9e-6 of max|ref|
# (2x3x200x232, partial mask).
REL = 1e-4

SHAPES = {"1x3x161x173": (1, 3, 161, 173),       # level 4 is exactly 11 x 11; the height pads at every level
          "2x3x200x232": (2, 3, 200, 232),
          "8x3x256x256": (8, 3, 256, 256),
          "1x3x768x512": (1, 3, 768, 512),
          "2x1x256x256": (2, 1, 256, 256)}
MASKS = ("ones", "blobs", "one_pixel", "one_transparent")


def _inputs(shape, mask_kind, seed=0):
    """X: bench.synthetic_rgba's colour planes; Y: X + noise; mask: see MASKS"""
    B, C, H, W = shape
    old = bench.IMG_H, bench.IMG_W
    bench.IMG_H, bench.IMG_W = H, W
    try:
        rgba = bench.synthetic_rgba(B, seed0=seed)
    finally:
        bench.IMG_H, bench.IMG_W = old
    g = torch.Generator().manual_seed(seed + 1)
    X = torch.rand(B, C, H, W, generator=g) * 0.3 + 0.7 * rgba[:, :C]
    Y = (X + 0.08 * torch.randn(B, C, H, W, generator=g)).clamp(0, 1)
    if mask_kind == "ones":
        mask = torch.ones(B, 1, H, W)
    elif mask_kind == "blobs":
        mask = rgba[:, 3:4].clone()
    elif mask_kind == "one_pixel":
        mask = torch.zeros(B, 1, H, W)
        mask[:, :, H // 3, W // 2] = 1.0                   # counted at some levels, not at all five
    else:
        mask = rgba[:, 3:4].clone()
        mask[0] = 0.0
    return X, Y, mask


def _ref_grads(X, Y, mask):
    """fp64 autograd through the oracle on the CPU"""
    Xr, Yr = X.double().requires_grad_(True), Y.double().requires_grad_(True)
    val = M.masked_ms_ssim(Xr, Yr, mask.double())
    gx, gy = torch.autograd.grad(val, (Xr, Yr))
    return float(val.detach()), gx, gy


def _oracle_on(dev, X, Y, mask):
    """the oracle's torch expressions in fp32 on `dev` (its helpers build their constants on the default device)"""
    with torch.device(dev):
        return M.masked_ms_ssim(X, Y, mask)


def _device_grads(pkg, dev, X, Y, mask, want_x, want_y):
    Xd, Yd = X.to(dev).requires_grad_(want_x), Y.to(dev).requires_grad_(want_y)
    val = pkg.masked_ms_ssim(Xd, Yd, mask.to(dev))
    val.backward()
    return val, Xd.grad, Yd.grad


@gpu
@pytest.mark.parametrize("mask_kind", MASKS)
@pytest.mark.parametrize("shape", list(SHAPES), ids=str)
def test_gradient_matches_fp64_autograd(pkg, cuda_dev, shape, mask_kind, record_property):
    B, C, H, W = SHAPES[shape]
    X, Y, mask = _inputs((B, C, H, W), mask_kind)
    ref_val, rx, ry = _ref_grads(X, Y, mask)
    # torch's own fp32 autograd through the same expressions, on the same device: the yardstick for the ratio
    X32, Y32 = X.to(cuda_dev).requires_grad_(True), Y.to(cuda_dev).requires_grad_(True)
    t32 = torch.autograd.grad(_oracle_on(cuda_dev, X32, Y32, mask.to(cuda_dev)), (X32, Y32))
    outside = (mask == 0).expand_as(X)
    report = {}
    for want_x, want_y in ((True, False), (False, True), (True, True)):
        val, gx, gy = _device_grads(pkg, cuda_dev, X, Y, mask, want_x, want_y)
        assert abs(float(val) - ref_val) < 1e-5, (float(val), ref_val)
        assert (gx is not None) == want_x and (gy is not None) == want_y
        for name, got, ref, tg in (("dX", gx, rx, t32[0]), ("dY", gy, ry, t32[1])):
            if got is None:
                continue
            got = got.cpu().double()
            assert torch.isfinite(got).all(), name
            assert torch.all(got[outside] == 0), f"{name}: nonzero gradient where the mask is 0"
            scale = float(ref.abs().max())
            err = (got - ref).abs()
            assert torch.all(err <= REL * scale), (name, want_x, want_y, float(err.max()), scale)
            if scale > 0:
                e32 = float((tg.cpu().double() - ref).abs().max()) / scale
                report[f"{name} x{int(want_x)}y{int(want_y)}"] = (float(err.max()) / scale, e32)
    if mask_kind == "one_pixel":
        assert ref_val == 0.0 and float(rx.abs().max()) == 0.0           # the fp64 gradient is exactly 0 ...
    if mask_kind == "one_transparent" and B > 1:
        val, gx, gy = _device_grads(pkg, cuda_dev, X, Y, mask, True, True)
        assert torch.all(gx[0] == 0) and torch.all(gy[0] == 0)
        assert float(rx[1:].abs().max()) > 0 and float(gx[1:].abs().max()) > 0
    for k, (ours, t) in report.items():
        record_property(k, f"{ours:.2e} of max|ref| (torch fp32 autograd {t:.2e}, ratio {ours / max(t, 1e-30):.2f})")
    print(shape, mask_kind, {k: f"{a:.2e} / torch fp32 {b:.2e}" for k, (a, b) in report.items()})


@gpu
def test_exact_properties(pkg, cuda_dev):
    X, Y, mask = _inputs((2, 3, 200, 232), "blobs", seed=5)
    Xd, Yd, md = X.to(cuda_dev).requires_grad_(True), Y.to(cuda_dev).requires_grad_(True), mask.to(cuda_dev)
    val = pkg.masked_ms_ssim(Xd, Yd, md)
    g1 = torch.autograd.grad(val, (Xd, Yd), retain_graph=True)
    g2 = torch.autograd.grad(val, (Xd, Yd))
    assert torch.equal(g1[0], g2[0]) and torch.equal(g1[1], g2[1])            # no atomics in the gradient path
    with torch.no_grad():
        plain = pkg.masked_ms_ssim(Xd, Yd, md)
    assert plain.grad_fn is None and val.grad_fn is not None
    assert abs(float(val) - float(plain)) < 1e-6                             # the forward's sums are atomic
    # neither input requires grad: the plain call, even with grad enabled
    assert pkg.masked_ms_ssim(Xd.detach(), Yd.detach(), md).grad_fn is None
    # a mask that requires grad gets none
    mg = md.clone().requires_grad_(True)
    pkg.masked_ms_ssim(Xd, Yd, mg).backward()
    assert mg.grad is None


def _metric_as_before(pkg, X, Y, mask, data_range=1.0, weights=(0.0448, 0.2856, 0.3001, 0.2363, 0.1333)):
    """masked_ms_ssim as it was before it became differentiable (what a no-grad call must still do)"""
    lib = pkg._abi.load()
    B, C, H, W = X.shape
    X, Y, m = X.contiguous(), Y.contiguous(), mask.reshape(B, H, W).contiguous()
    vals = []
    st = pkg._abi.stream_handle()
    with torch.cuda.device(X.device):
        for lvl in range(len(weights)):
            sums = torch.empty(B, C, 2, device=X.device, dtype=torch.float32)
            cnt = torch.empty(B, device=X.device, dtype=torch.float32)
            pkg._abi.check(lib.ms_ssim_level_forward(X.data_ptr(), Y.data_ptr(), m.data_ptr(), B, C, H, W, float(data_range),
                                                     sums.data_ptr(), cnt.data_ptr(), st), "ms_ssim_level_forward")
            per = sums / (cnt.view(B, 1, 1) + 1e-10)
            if lvl < len(weights) - 1:
                vals.append(torch.relu(per[..., 1]))
                Hp, Wp = (H + 2 * (H % 2) - 2) // 2 + 1, (W + 2 * (W % 2) - 2) // 2 + 1
                Xo = torch.empty(B, C, Hp, Wp, device=X.device, dtype=torch.float32)
                Yo, Mo = torch.empty_like(Xo), torch.empty(B, Hp, Wp, device=X.device, dtype=torch.float32)
                pkg._abi.check(lib.ms_ssim_pool_forward(X.data_ptr(), Y.data_ptr(), m.data_ptr(), B, C, H, W, Xo.data_ptr(),
                                                        Yo.data_ptr(), Mo.data_ptr(), st), "ms_ssim_pool_forward")
                X, Y, m, H, W = Xo, Yo, Mo, Hp, Wp
            else:
                vals.append(torch.relu(per[..., 0]))
    w = torch.tensor(weights, device=X.device, dtype=torch.float32).view(-1, 1, 1)
    return torch.prod(torch.stack(vals, 0) ** w, dim=0).mean()


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return out, names


@gpu
def test_no_grad_call_launches_what_it_did_before(pkg, cuda_dev):
    X, Y, mask = (t.to(cuda_dev) for t in _inputs((2, 3, 200, 232), "blobs", seed=7))
    _metric_as_before(pkg, X, Y, mask), pkg.masked_ms_ssim(X, Y, mask)       # warm-up
    before, k_before = _kernels(lambda: _metric_as_before(pkg, X, Y, mask))
    now, k_now = _kernels(lambda: pkg.masked_ms_ssim(X, Y, mask))
    with torch.no_grad():
        Xg = X.clone().requires_grad_(True)
        nograd, k_nograd = _kernels(lambda: pkg.masked_ms_ssim(Xg, Y, mask))
    assert k_now == k_before and k_nograd == k_before, (k_before, k_now, k_nograd)
    assert sum("ms_ssim_level_kernel" in k for k in k_before) == 5
    assert not any("bwd" in k for k in k_before)
    assert abs(float(now) - float(before)) < 1e-6 and abs(float(nograd) - float(before)) < 1e-6   # atomic sums


def _syncs(fn):
    """where the synchronising CUDA calls torch reports while fn runs were made (file:line)"""
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            fn()
        finally:
            torch.cuda.set_sync_debug_mode("default")
    return [f"{os.path.basename(w.filename)}:{w.lineno}" for w in caught
            if "called a synchronizing CUDA operation" in str(w.message)]


@gpu
def test_five_backward_launches_and_no_synchronisation(pkg, lib, cuda_dev, monkeypatch):
    X, Y, mask = (t.to(cuda_dev) for t in _inputs((2, 3, 256, 256), "blobs", seed=3))
    for want in ((True, False), (False, True), (True, True)):
        Xd, Yd = X.clone().requires_grad_(want[0]), Y.clone().requires_grad_(want[1])
        pkg.masked_ms_ssim(Xd, Yd, mask).backward()                          # warm-up
        calls = []
        real = lib.ms_ssim_level_backward

        def spy(*args):
            status = real(*args)
            calls.append((args[5], args[6], args[12] is not None, args[13] is not None, status))   # H, W, dX, dY
            return status

        monkeypatch.setattr(lib, "ms_ssim_level_backward", spy)
        loss = 1 - pkg.masked_ms_ssim(Xd, Yd, mask)
        torch.cuda.synchronize()
        syncs = _syncs(loss.backward)
        monkeypatch.setattr(lib, "ms_ssim_level_backward", real)
        assert syncs == [], syncs
        assert [(h, w) for h, w, *_ in calls] == [(16, 16), (32, 32), (64, 64), (128, 128), (256, 256)], calls
        assert all(c[2] == want[0] and c[3] == want[1] and c[4] == 0 for c in calls), calls
    # the detector sees a synchronisation made inside a backward: torch.prod's reads its zero count on the host
    v = torch.rand(5, 4, device=cuda_dev, requires_grad=True)
    torch.prod(v, dim=0).sum().backward()
    assert _syncs(lambda: torch.prod(v, dim=0).sum().backward())


def test_status_codes_before_any_launch(lib):
    one = ctypes.c_void_p(256)
    bwd = lib.ms_ssim_level_backward
    args = [one, one, one, 2, 3, 64, 64, 1.0, one, one, None, None, one, one, None]
    assert len(bwd.argtypes) == len(args)
    for i in (0, 1, 2, 8, 9):                                 # X, Y, mask, grad, counts
        a = list(args)
        a[i] = None
        assert bwd(*a) == -1, i
    for B, C in ((-1, 3), (2, 0), (2, -3)):
        a = list(args)
        a[3], a[4] = B, C
        assert bwd(*a) == -1, (B, C)
    for H, W in ((10, 64), (64, 10), (0, 64)):
        a = list(args)
        a[5], a[6] = H, W
        assert bwd(*a) == -2, (H, W)
    a = list(args)
    a[3] = 0
    assert bwd(*a) == 0                                       # an empty batch launches nothing
    a = list(args)
    a[12] = a[13] = None
    assert bwd(*a) == 0                                       # no output asked for: nothing to do


def test_binding_matches_header(pkg):
    text = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "mwa_b200.h")).read()
    assert "MWA_API int ms_ssim_level_backward(" in text
    assert "ms_ssim_level_backward" in pkg._abi.EXPORTED_SYMBOLS


@gpu
def test_training_step_with_ms_ssim_distortion(pkg, cuda_dev, model_keys):
    """one step of the codec with loss = 1 - masked_ms_ssim(x_hat, image, mask) + bpp: its parameter gradients equal
    those of the same step with the oracle's MS-SSIM run in fp32 on the device"""
    cfg = next(iter(G.MODEL_CASES.values()))
    net = pkg.RGBACodec().train()
    net.load_state_dict(G.model_state(model_keys, cfg["seed"]), strict=False)
    net = net.to(cuda_dev)
    old = bench.IMG_H, bench.IMG_W
    bench.IMG_H = bench.IMG_W = 256
    try:
        rgba = bench.synthetic_rgba(2, seed0=21).to(cuda_dev)
    finally:
        bench.IMG_H, bench.IMG_W = old
    image, mask = rgba[:, :3].contiguous(), rgba[:, 3:4].contiguous()

    def step(ms_ssim):
        net.zero_grad(set_to_none=True)
        me = net.EncMakeMask(mask)
        x_hat, _, bpp, _, _ = net(image, mask, mask, me[0], me[1], me[2], me[3])
        loss = 1 - ms_ssim(x_hat, image, mask) + bpp
        loss.backward()
        return float(loss), {n: p.grad.detach().clone() for n, p in net.named_parameters() if p.grad is not None}

    l_dev, g_dev = step(pkg.masked_ms_ssim)
    l_ref, g_ref = step(lambda a, b, m: _oracle_on(cuda_dev, a, b, m))
    assert abs(l_dev - l_ref) < 1e-5, (l_dev, l_ref)
    assert g_dev.keys() == g_ref.keys() and len(g_dev) > 100
    worst = 0.0
    for n, gr in g_ref.items():
        scale = float(gr.abs().max())
        err = float((g_dev[n] - gr).abs().max())
        assert err <= 2e-3 * scale + 1e-12, (n, err, scale)
        worst = max(worst, err / scale if scale > 0 else 0.0)
    print("training step: largest max|err| / max|ref| over the parameter gradients", f"{worst:.2e}")
