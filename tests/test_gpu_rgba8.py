"""8-bit RGBA images of any size (csrc/rgba8.cu, <package>/rgba8.py, codec.AutoEncoder.compress_rgba8 / decompress_rgba8;
DESIGN.md 4.8).  The ingest and egress kernels are held bit for bit to torch expressions; the smallest geometries that
padding produces (64 x 64: an 8 x 8 latent, a 1 x 1 z) are held to the CPU oracle with tests/test_gpu_model.py's criteria;
padding must be invisible in the bitstream (a multiple of 64 is coded exactly as `compress` codes its planes, and an image
padded by hand with transparent pixels gives the same strings), and decompress_rgba8 must return exactly the torch egress
of the encoder-side reconstruction.  Argument checks run without a GPU."""
import ctypes
import os
import warnings

import pytest
import torch
import torch.nn.functional as F

from oracle import golden_cases as G
from oracle import ref_model as M

gpu = pytest.mark.gpu
RTOL, ATOL = 1e-3, 1e-4
KERNEL_SIZES = [(1, 1), (1, 1000), (63, 65), (64, 64), (511, 767), (2160, 3840)]


def _padded(n):
    return -(-n // 64) * 64


def _image8(B, H, W, seed):
    """uint8 (B, H, W, 4): smooth colour + noise, soft alpha with fully transparent 16 x 16 blocks.  The colour is NOT
    premultiplied: under alpha 0 it is arbitrary, and the ingest must zero it."""
    g = torch.Generator().manual_seed(seed)
    yy = torch.linspace(0, 1, H).view(1, H, 1)
    xx = torch.linspace(0, 1, W).view(1, 1, W)
    rgb = torch.stack([0.5 + 0.4 * torch.sin(6.0 * xx + 3.0 * yy), 0.5 + 0.4 * torch.cos(5.0 * yy - 2.0 * xx),
                       0.5 + 0.3 * torch.sin(9.0 * xx * yy + 1.0)], -1)
    rgb = (rgb + 0.08 * torch.randn(B, H, W, 3, generator=g)).clamp(0, 1)
    keep = torch.rand(B, (H + 15) // 16, (W + 15) // 16, generator=g) >= 0.35
    keep = keep.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :H, :W]
    alpha = (0.3 + 0.7 * torch.rand(B, H, W, generator=g)) * keep
    return (torch.cat([rgb, alpha[..., None]], -1) * 255).round().to(torch.uint8)


def _random8(B, H, W, C, seed):
    """uniform bytes, alpha zero on ~30 % of the pixels"""
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, 256, (B, H, W, C), generator=g, dtype=torch.uint8)
    t[..., -1] *= (torch.rand(B, H, W, generator=g) >= 0.3).to(torch.uint8)
    return t


def _ingest_ref(t):
    """the torch expression, on the CPU: there `/ 255` is an IEEE division (on CUDA, torch multiplies by 1/255, which
    differs on 126 of the 256 byte values).  Made contiguous: the permute leaves the planes channels-last in memory."""
    B, H, W, C = t.shape
    f = F.pad(t.permute(0, 3, 1, 2).float() / 255, (0, _padded(W) - W, 0, _padded(H) - H))
    alpha = f[:, C - 1:C].contiguous()
    return ((f[:, :3] * (alpha > 0)).contiguous() if C == 4 else None), alpha


def _egress_ref(x_hat, alpha8):
    B, H, W = alpha8.shape
    rgb = (x_hat[:, :, :H, :W].nan_to_num(0).clamp(0, 1) * 255).round().to(torch.uint8)
    rgb = rgb * (alpha8 > 0)[:, None].to(torch.uint8)
    return torch.cat([rgb.permute(0, 2, 3, 1), alpha8[..., None]], -1)


def _specials(B, H, W, seed):
    """fp32 x_hat (B, 3, Hp, Wp) in [-0.5, 1.5] with NaN, +-Inf, exact 0 / 1 and k / 255 values sprinkled in"""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, _padded(H), _padded(W), generator=g) * 2 - 0.5
    pick = torch.rand(x.shape, generator=g)
    x[pick < 0.02] = float("nan")
    x[(pick >= 0.02) & (pick < 0.03)] = float("inf")
    x[(pick >= 0.03) & (pick < 0.04)] = float("-inf")
    x[(pick >= 0.04) & (pick < 0.05)] = 1.0
    x[(pick >= 0.05) & (pick < 0.06)] = 0.0
    k = (pick >= 0.06) & (pick < 0.1)
    x[k] = torch.randint(0, 256, (int(k.sum()),), generator=g).float() / 255
    return x


# ------------------------------------------------------------------------------------------------ CPU: arguments
def test_status_codes_before_any_launch(lib):
    one, odd = ctypes.c_void_p(256), ctypes.c_void_p(258)
    ing, eg = lib.rgba8_ingest, lib.rgba8_egress
    # null pointers
    assert ing(None, one, one, 1, 8, 8, 4, None) == -1
    assert ing(one, one, None, 1, 8, 8, 4, None) == -1
    assert ing(one, None, one, 1, 8, 8, 4, None) == -1                   # C = 4 needs the image planes
    assert eg(None, one, one, 1, 8, 8, None) == -1
    assert eg(one, None, one, 1, 8, 8, None) == -1
    assert eg(one, one, None, 1, 8, 8, None) == -1
    # sizes and channels
    for B, H, W in ((-1, 8, 8), (1, 0, 8), (1, 8, 0), (1, -5, 8), (1, 2 ** 31 - 1, 1)):
        assert ing(one, one, one, B, H, W, 4, None) == -1, (B, H, W)
        assert eg(one, one, one, B, H, W, None) == -1, (B, H, W)
    for C in (0, 2, 3, 5, -4):
        assert ing(one, one, one, 1, 8, 8, C, None) == -1, C
    # B * Hp * Wp * 48 < 2^31: 10922 images of 64 x 64 are the most, 8192 x 8192 is too large even alone
    assert ing(one, one, one, 10923, 64, 64, 4, None) == -1
    assert ing(one, one, one, 10923, 1, 1, 1, None) == -1
    assert eg(one, one, one, 10923, 64, 64, None) == -1
    assert ing(one, one, one, 1, 8192, 8192, 4, None) == -1
    assert eg(one, one, one, 1, 8192, 8192, None) == -1
    assert ing(one, one, one, 1, 4096, 10881, 4, None) == -1           # Wp = 10944: 4096 * 10944 * 48 = 2^31 + 4.2e6
    # alignment: fp32 planes 16 bytes, RGBA buffers 4 bytes
    assert ing(one, one, odd, 1, 8, 8, 4, None) == -3
    assert ing(one, odd, one, 1, 8, 8, 4, None) == -3
    assert ing(odd, one, one, 1, 8, 8, 4, None) == -3
    assert eg(odd, one, one, 1, 8, 8, None) == -3
    assert eg(one, one, odd, 1, 8, 8, None) == -3
    # an empty batch launches nothing, whatever the pointers
    assert ing(None, None, None, 0, 8, 8, 4, None) == 0
    assert ing(None, None, None, 0, 8, 8, 1, None) == 0
    assert eg(None, None, None, 0, 8, 8, None) == 0


def test_python_wrappers_reject_bad_inputs(pkg):
    good = torch.zeros(2, 5, 7, 4, dtype=torch.uint8)
    with pytest.raises(pkg.MwaB200Error, match="uint8"):
        pkg.rgba8_ingest(good.float())
    for bad in (torch.zeros(5, 7, dtype=torch.uint8), torch.zeros(2, 5, 7, 3, dtype=torch.uint8),
                torch.zeros(1, 2, 5, 7, 4, dtype=torch.uint8), torch.zeros(1, 0, 7, 4, dtype=torch.uint8),
                torch.zeros(1, 5, 0, 4, dtype=torch.uint8)):
        with pytest.raises(ValueError):
            pkg.rgba8_ingest(bad)
    with pytest.raises(ValueError, match="contiguous"):
        pkg.rgba8_ingest(torch.zeros(2, 7, 5, 4, dtype=torch.uint8).transpose(1, 2))
    with pytest.raises(ValueError):
        pkg.rgba8_ingest(good.numpy())
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        pkg.rgba8._check_size(1, 8192, 8192)
    pkg.rgba8._check_size(10922, 64, 64)
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        pkg.rgba8._check_size(10923, 64, 64)
    with pytest.raises(pkg.MwaB200Error, match="CUDA"):
        pkg.rgba8_egress(torch.zeros(1, 3, 64, 64), torch.zeros(1, 5, 7, dtype=torch.uint8))


def test_codec_rejects_bad_arguments_before_any_launch(pkg):
    net = pkg.RGBACodec().eval()
    img = torch.zeros(63, 65, 4, dtype=torch.uint8)
    with pytest.raises(ValueError, match="coder"):
        net.compress_rgba8(img, coder="gpu")
    with pytest.raises(ValueError):
        net.compress_rgba8(img[..., :1].contiguous())                   # alpha alone is not an image
    alpha8 = torch.zeros(1, 63, 65, dtype=torch.uint8)
    strings = [[b"\0" * 8], [b"\0" * 8]]
    for shape in ((2, 2), (1, 1), (1, 2, 1)):
        with pytest.raises(ValueError, match="shape"):
            net.decompress_rgba8(strings, shape, alpha8)
    with pytest.raises(ValueError, match="images"):
        net.decompress_rgba8([[b"\0" * 8] * 2, [b"\0" * 8] * 2], (1, 2), alpha8)
    with pytest.raises(ValueError, match="contiguous"):
        net.decompress_rgba8(strings, (1, 2), torch.zeros(1, 65, 63, dtype=torch.uint8).transpose(1, 2))
    with pytest.raises(pkg.MwaB200Error, match="uint8"):
        net.decompress_rgba8(strings, (1, 2), alpha8.float())


# ------------------------------------------------------------------------------------------------ GPU: kernels
@gpu
@pytest.mark.parametrize("B", [0, 1, 3])
@pytest.mark.parametrize("H,W", KERNEL_SIZES)
def test_ingest_equals_torch(pkg, cuda_dev, B, H, W):
    for C in (4, 1):
        t = _random8(B, H, W, C, seed=H * 7 + W + B)
        image, alpha, size = pkg.rgba8_ingest(t.to(cuda_dev))
        ref_image, ref_alpha = _ingest_ref(t)
        assert size == (H, W)
        assert alpha.shape == (B, 1, _padded(H), _padded(W)) and alpha.dtype == torch.float32
        assert torch.equal(alpha.cpu(), ref_alpha) and not torch.signbit(alpha).any()
        if C == 4:
            assert image.shape == (B, 3, _padded(H), _padded(W))
            assert torch.equal(image.cpu(), ref_image) and not torch.signbit(image).any()
        else:
            assert image is None


@gpu
@pytest.mark.parametrize("B", [0, 1, 3])
@pytest.mark.parametrize("H,W", KERNEL_SIZES)
def test_egress_equals_torch(pkg, cuda_dev, B, H, W):
    x = _specials(B, H, W, seed=H + 3 * W + B)
    a8 = _random8(B, H, W, 1, seed=H + W + 11 * B)[..., 0].contiguous()
    got = pkg.rgba8_egress(x.to(cuda_dev), a8.to(cuda_dev))
    assert got.shape == (B, H, W, 4) and got.dtype == torch.uint8 and got.is_cuda
    assert torch.equal(got.cpu(), _egress_ref(x, a8))


@gpu
def test_host_inputs_side_stream_and_graph_capture(pkg, cuda_dev):
    B, H, W = 3, 63, 65
    t = _random8(B, H, W, 4, seed=5)
    x = _specials(B, H, W, seed=6)
    a8 = t[..., 3].contiguous()
    ref_image, ref_alpha = _ingest_ref(t)
    ref_out = _egress_ref(x, a8)
    # host inputs, pageable and pinned: copied to the device once
    for src in (t, t.pin_memory()):
        image, alpha, _ = pkg.rgba8_ingest(src)
        assert image.is_cuda and torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha)
    assert torch.equal(pkg.rgba8_egress(x.to(cuda_dev), a8.pin_memory()).cpu(), ref_out)
    td, xd, ad = t.to(cuda_dev), x.to(cuda_dev), a8.to(cuda_dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        image, alpha, _ = pkg.rgba8_ingest(td)
        out = pkg.rgba8_egress(xd, ad)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha)
    assert torch.equal(out.cpu(), ref_out)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        image, alpha, _ = pkg.rgba8_ingest(td)
        out = pkg.rgba8_egress(xd, ad)
    for _ in range(2):
        for o in (image, alpha):
            o.fill_(-1.0)
        out.fill_(7)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha)
        assert torch.equal(out.cpu(), ref_out)


# ------------------------------------------------------------------------------------------------ GPU: the codec
@pytest.fixture
def net(pkg, cuda_dev, model_keys):
    """the codec on G.model_state weights, with cuDNN (the 3-channel convolutions) held to deterministic algorithms: the
    exact comparisons below run the same layers in separate calls"""
    prev = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    model = pkg.RGBACodec().eval()
    model.load_state_dict(G.model_state(model_keys, 61), strict=False)
    try:
        yield model.to(cuda_dev)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev


@gpu
@pytest.mark.parametrize("H,W", [(64, 64), (64, 192), (192, 64)])
def test_smallest_geometries_match_the_oracle(cuda_dev, model_keys, net, H, W):
    """64 x 64: 2 x 2 windows of 8 x 8 at 1/4 scale and of 4 x 4 at 1/8 scale, an 8 x 8 latent, a 1 x 1 z"""
    seed = 61
    p = G.model_inputs(dict(B=1, H=H, W=W, drop=0.35, seed=seed + H + W))
    with torch.no_grad():
        r = {k: v.cpu() for k, v in net.detail(*(p[k].to(cuda_dev) for k in ("image", "alpha", "reconmask"))).items()}
    w = G.model_state(model_keys, seed)
    with torch.no_grad():
        o = M.rgb_forward(w, p["image"], p["alpha"], p["reconmask"])
    assert r["z"].shape == (1, 192, H // 64, W // 64) and r["y"].shape == (1, 80, H // 8, W // 8)
    torch.testing.assert_close(r["y"], o["y"], rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(r["z"], o["z"], rtol=RTOL, atol=ATOL)
    # rounded latents: equal except genuine .5 ties (tests/test_gpu_model.py's rule)
    flipped = (r["y_hat"] - o["y_hat"]).abs() > 0.5
    frac = float(flipped.float().mean())
    assert frac < 2e-3, frac
    sl = r["y_hat"].shape[1] // 10
    first_flip = next((i for i in range(10) if bool(flipped[:, i * sl:(i + 1) * sl].any())), 10)
    if first_flip > 0:
        torch.testing.assert_close(r["y_hat"][:, :first_flip * sl], o["y_hat"][:, :first_flip * sl], rtol=RTOL, atol=ATOL)
    if first_flip < 10:
        s = slice(first_flip * sl, (first_flip + 1) * sl)
        resid = o["y"][:, s] - o["means"][:, s]
        tie = (resid - torch.floor(resid) - 0.5).abs()
        assert float(tie[flipped[:, s]].max()) < 2e-3
    if frac == 0.0:
        torch.testing.assert_close(r["x_hat"], o["x_hat"], rtol=RTOL, atol=ATOL)
    else:
        assert float(((r["x_hat"] - o["x_hat"]).abs() > ATOL + RTOL * o["x_hat"].abs()).float().mean()) < 0.05


@gpu
def test_multiple_of_64_is_coded_as_compress_codes_its_planes(cuda_dev, net):
    t = _image8(2, 192, 256, seed=3)
    image, alpha = (v.to(cuda_dev) for v in _ingest_ref(t))
    for coder in ("host", "device"):
        with torch.no_grad():
            got = net.compress_rgba8(t.to(cuda_dev), coder=coder)
            want = net.compress(image, alpha, coder=coder)
        assert got["size"] == (192, 256) and tuple(got["shape"]) == tuple(want["shape"]) == (3, 4)
        assert got["strings"] == want["strings"], coder


@gpu
@pytest.mark.parametrize("H,W", [(63, 65), (511, 767)])
def test_padding_is_transparent(cuda_dev, net, H, W):
    t = _image8(1, H, W, seed=H + W)
    by_hand = torch.zeros(1, _padded(H), _padded(W), 4, dtype=torch.uint8)
    by_hand[:, :H, :W] = t
    for coder in ("host", "device"):
        with torch.no_grad():
            a = net.compress_rgba8(t.to(cuda_dev), coder=coder)
            b = net.compress_rgba8(by_hand.to(cuda_dev), coder=coder)
            assert a["strings"] == b["strings"] and tuple(a["shape"]) == tuple(b["shape"]), coder
            rec_a = net.decompress_rgba8(a["strings"], a["shape"], t[..., 3].contiguous().to(cuda_dev))
            rec_b = net.decompress_rgba8(b["strings"], b["shape"], by_hand[..., 3].contiguous().to(cuda_dev))
        assert rec_a.shape == (1, H, W, 4)
        assert torch.equal(rec_a, rec_b[:, :H, :W]), coder


@gpu
@pytest.mark.parametrize("H,W", [(63, 65), (511, 767), (2160, 3840)])
def test_round_trip_equals_torch_egress_of_the_forward(pkg, cuda_dev, net, H, W):
    t = _image8(1, H, W, seed=2 * H + W)
    td = t.to(cuda_dev)
    a8 = t[..., 3].contiguous()
    image, alpha, _ = pkg.rgba8_ingest(td)
    with torch.no_grad():
        me = net.EncMakeMask(alpha)
        x_hat = net(image, alpha, alpha, me[0], me[1], me[2], me[3])[0]
    want = _egress_ref(x_hat.cpu(), a8)
    for coder, lanes in (("host", None), ("device", None), ("device", 7)):
        with torch.no_grad():
            out = net.compress_rgba8(td, coder=coder, lanes=lanes)
            assert out["size"] == (H, W) and tuple(out["shape"]) == (_padded(H) // 64, _padded(W) // 64)
            rec = net.decompress_rgba8(out["strings"], out["shape"], a8.to(cuda_dev))
        assert rec.shape == (1, H, W, 4) and rec.dtype == torch.uint8
        rec = rec.cpu()
        assert torch.equal(rec, want), (coder, lanes)
        assert torch.equal(rec[..., 3], a8)
        assert not rec[..., :3][a8 == 0].any()


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
def test_synchronisation_counts(pkg, cuda_dev, net):
    t = _image8(2, 63, 65, seed=9).to(cuda_dev)
    a8 = t[..., 3].contiguous()
    image, alpha, _ = pkg.rgba8_ingest(t)
    with torch.no_grad():
        for coder in ("host", "device"):                          # warm-up: tables on the device, kernels loaded
            out = net.compress_rgba8(t, coder=coder)
            net.compress(image, alpha, coder=coder)
            net.decompress_rgba8(out["strings"], out["shape"], a8)
        dev_out = net.compress_rgba8(t, coder="device")
        torch.cuda.synchronize()
        on_dev = _syncs(lambda: net.decompress_rgba8(dev_out["strings"], dev_out["shape"], a8))
        assert len(on_dev) <= 1, on_dev
        for coder in ("host", "device"):
            torch.cuda.synchronize()
            eight = _syncs(lambda: net.compress_rgba8(t, coder=coder))
            planes = _syncs(lambda: net.compress(image, alpha, coder=coder))
            assert len(eight) <= len(planes), (coder, eight, planes)
