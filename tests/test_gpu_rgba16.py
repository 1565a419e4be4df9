"""16-bit RGBA images of any size (csrc/rgba8.cu's uint16 instantiations, <package>/rgba8.py's rgba16_ingest / rgba16_egress,
codec.AutoEncoder.compress_rgba16 / decompress_rgba16; DESIGN.md 4.8).  The kernels are held bit for bit to torch
expressions computed on the CPU in int32 / fp32 (no reference depends on uint16 arithmetic); for 8-bit images v the
16-bit path must see 257 * v exactly as the 8-bit path sees v, planes and strings alike; strings decode at either bit
depth.  Argument checks run without a GPU."""
import ctypes
import os
import warnings

import pytest
import torch
import torch.nn.functional as F

from oracle import golden_cases as G

gpu = pytest.mark.gpu
FULL = 65535
KERNEL_SIZES = [(1, 1), (5, 7), (63, 65), (65, 63), (256, 257)]


def _padded(n):
    return -(-n // 64) * 64


def _i32(t):
    """a uint16 result as int32 on the CPU, where comparisons need no uint16 op support"""
    return t.cpu().to(torch.int32)


def _u16(t):
    return t.to(torch.int32).to(torch.uint16)


def _zeros16(n, device):
    """uint16 zeros on the device, written as int16: torch has few CUDA kernels for uint16"""
    return torch.zeros(n, dtype=torch.int16, device=device).view(torch.uint16)


def _random16(B, H, W, C, seed):
    """uniform uint16 samples, alpha zero on ~30 % of the pixels; where there are at least 65536 pixels, the first 65536
    alphas of the batch are a permutation of every uint16 value"""
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, FULL + 1, (B, H, W, C), generator=g, dtype=torch.int32)
    t[..., -1] *= (torch.rand(B, H, W, generator=g) >= 0.3).to(torch.int32)
    if B * H * W >= FULL + 1:
        t.view(-1, C)[:FULL + 1, -1] = torch.randperm(FULL + 1, generator=g, dtype=torch.int32)
    return _u16(t)


def _image8(B, H, W, seed):
    """uint8 (B, H, W, 4): smooth colour + noise, soft alpha with fully transparent 16 x 16 blocks, colour not premultiplied"""
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


def _image16(B, H, W, seed):
    """the same kind of image at 16 bits, with values that no 8-bit image has"""
    g = torch.Generator().manual_seed(seed + 1)
    t = _image8(B, H, W, seed).to(torch.int32) * 257 + torch.randint(-128, 129, (B, H, W, 4), generator=g, dtype=torch.int32)
    t = t.clamp(0, FULL)
    t[..., 3] *= (t[..., 3] > 200).to(torch.int32)                  # keep the transparent blocks transparent
    return _u16(t)


def _times257(t8):
    return _u16(t8.to(torch.int32) * 257)


def _ingest_ref(t):
    """the torch expression on the CPU, where `/ 65535` is an IEEE division"""
    B, H, W, C = t.shape
    f = F.pad(t.to(torch.int32).permute(0, 3, 1, 2).float() / FULL, (0, _padded(W) - W, 0, _padded(H) - H))
    alpha = f[:, C - 1:C].contiguous()
    return ((f[:, :3] * (alpha > 0)).contiguous() if C == 4 else None), alpha


def _egress_ref(x_hat, alpha16):
    """int32 (B, H, W, 4): rint(clamp(x, 0, 1) * 65535) in fp32 where alpha > 0, else 0; A = alpha"""
    B, H, W = alpha16.shape
    a = alpha16.to(torch.int32)
    rgb = (x_hat[:, :, :H, :W].nan_to_num(0).clamp(0, 1) * FULL).round().to(torch.int32) * (a > 0)[:, None]
    return torch.cat([rgb.permute(0, 2, 3, 1), a[..., None]], -1)


def _specials(B, H, W, seed):
    """fp32 x_hat (B, 3, Hp, Wp) in [-0.5, 1.5] with NaN, +-Inf, exact 0 / 1 and k / 65535 values sprinkled in"""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(B, 3, _padded(H), _padded(W), generator=g) * 2 - 0.5
    pick = torch.rand(x.shape, generator=g)
    x[pick < 0.02] = float("nan")
    x[(pick >= 0.02) & (pick < 0.03)] = float("inf")
    x[(pick >= 0.03) & (pick < 0.04)] = float("-inf")
    x[(pick >= 0.04) & (pick < 0.05)] = 1.0
    x[(pick >= 0.05) & (pick < 0.06)] = 0.0
    k = (pick >= 0.06) & (pick < 0.1)
    x[k] = torch.randint(0, FULL + 1, (int(k.sum()),), generator=g).float() / FULL
    return x


# ------------------------------------------------------------------------------------------------ CPU: arguments
def test_status_codes_before_any_launch(lib):
    one, odd, four, two = ctypes.c_void_p(256), ctypes.c_void_p(257), ctypes.c_void_p(260), ctypes.c_void_p(258)
    ing, eg = lib.rgba16_ingest, lib.rgba16_egress
    # null pointers
    assert ing(None, one, one, 1, 8, 8, 4, None) == -1
    assert ing(None, None, one, 1, 8, 8, 1, None) == -1
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
    # B * Hp * Wp * 48 < 2^31: 10922 images of 64 x 64 pass the size guard (and stop at the misaligned buffer), 10923 and
    # one 8192 x 8192 image do not
    assert ing(four, one, one, 10922, 64, 64, 4, None) == -3
    assert eg(one, one, four, 10922, 64, 64, None) == -3
    assert ing(one, one, one, 10923, 64, 64, 4, None) == -1
    assert ing(one, one, one, 10923, 1, 1, 1, None) == -1
    assert eg(one, one, one, 10923, 64, 64, None) == -1
    assert ing(one, one, one, 1, 8192, 8192, 4, None) == -1
    assert eg(one, one, one, 1, 8192, 8192, None) == -1
    # alignment: fp32 planes 16 bytes, RGBA buffers 8 bytes, alpha-only buffers 2 bytes
    assert ing(one, one, two, 1, 8, 8, 4, None) == -3
    assert ing(one, two, one, 1, 8, 8, 4, None) == -3
    assert ing(four, one, one, 1, 8, 8, 4, None) == -3
    assert ing(two, one, one, 1, 8, 8, 4, None) == -3
    assert ing(odd, None, one, 1, 8, 8, 1, None) == -3
    assert eg(two, one, one, 1, 8, 8, None) == -3
    assert eg(one, one, four, 1, 8, 8, None) == -3
    assert eg(one, odd, one, 1, 8, 8, None) == -3
    # an empty batch launches nothing, whatever the pointers
    assert ing(None, None, None, 0, 8, 8, 4, None) == 0
    assert ing(None, None, None, 0, 8, 8, 1, None) == 0
    assert eg(None, None, None, 0, 8, 8, None) == 0


def test_python_wrappers_reject_bad_inputs(pkg):
    good16 = torch.zeros(2, 5, 7, 4, dtype=torch.uint16)
    good8 = torch.zeros(2, 5, 7, 4, dtype=torch.uint8)
    for bad in (good8, good16.to(torch.int32), good16.to(torch.int16), good8.float()):
        with pytest.raises(pkg.MwaB200Error, match="must be uint16"):
            pkg.rgba16_ingest(bad)
    with pytest.raises(pkg.MwaB200Error, match="must be uint8"):
        pkg.rgba8_ingest(good16)
    for shape in ((5, 7), (2, 5, 7, 3), (1, 2, 5, 7, 4), (1, 0, 7, 4), (1, 5, 0, 4)):
        with pytest.raises(ValueError):
            pkg.rgba16_ingest(torch.zeros(shape, dtype=torch.uint16))
    with pytest.raises(ValueError, match="contiguous"):
        pkg.rgba16_ingest(torch.zeros(2, 7, 5, 4, dtype=torch.uint16).transpose(1, 2))
    with pytest.raises(ValueError):
        pkg.rgba16_ingest(good16.numpy())
    with pytest.raises(pkg.MwaB200Error, match="CUDA"):
        pkg.rgba16_egress(torch.zeros(1, 3, 64, 64), torch.zeros(1, 5, 7, dtype=torch.uint16))


@gpu
def test_egress_rejects_bad_alpha_before_any_launch(pkg, cuda_dev):
    """the alpha must be contiguous (B, H, W) of the entry point's dtype and fit x_hat"""
    x = torch.zeros(1, 3, 64, 64, device=cuda_dev)
    launches = pkg._abi.launch_count
    with pytest.raises(ValueError, match="uint16"):
        pkg.rgba16_egress(x, torch.zeros(1, 5, 7, dtype=torch.uint8))
    with pytest.raises(ValueError, match="uint8"):
        pkg.rgba8_egress(x, torch.zeros(1, 5, 7, dtype=torch.uint16))
    with pytest.raises(ValueError, match="contiguous"):
        pkg.rgba16_egress(x, torch.zeros(1, 7, 5, dtype=torch.uint16).transpose(1, 2))
    with pytest.raises(ValueError):
        pkg.rgba16_egress(x, torch.zeros(5, 7, dtype=torch.uint16))
    with pytest.raises(ValueError, match="x_hat"):
        pkg.rgba16_egress(x, torch.zeros(1, 5, 65, dtype=torch.uint16))
    assert pkg._abi.launch_count == launches


def test_codec_rejects_bad_arguments_before_any_launch(pkg):
    net = pkg.RGBACodec().eval()
    img = torch.zeros(63, 65, 4, dtype=torch.uint16)
    with pytest.raises(ValueError, match="coder"):
        net.compress_rgba16(img, coder="gpu")
    with pytest.raises(ValueError):
        net.compress_rgba16(img[..., :1].contiguous())                  # alpha alone is not an image
    with pytest.raises(pkg.MwaB200Error, match="uint16"):
        net.compress_rgba16(img.to(torch.int32).to(torch.uint8))
    with pytest.raises(pkg.MwaB200Error, match="uint8"):
        net.compress_rgba8(img)
    alpha16 = torch.zeros(1, 63, 65, dtype=torch.uint16)
    strings = [[b"\0" * 8], [b"\0" * 8]]
    for shape in ((2, 2), (1, 1), (1, 2, 1)):
        with pytest.raises(ValueError, match="shape"):
            net.decompress_rgba16(strings, shape, alpha16)
    with pytest.raises(ValueError, match="images"):
        net.decompress_rgba16([[b"\0" * 8] * 2, [b"\0" * 8] * 2], (1, 2), alpha16)
    with pytest.raises(ValueError, match="contiguous"):
        net.decompress_rgba16(strings, (1, 2), torch.zeros(1, 65, 63, dtype=torch.uint16).transpose(1, 2))
    with pytest.raises(pkg.MwaB200Error, match="uint16"):
        net.decompress_rgba16(strings, (1, 2), torch.zeros(1, 63, 65, dtype=torch.uint8))
    with pytest.raises(pkg.MwaB200Error, match="uint8"):
        net.decompress_rgba8(strings, (1, 2), alpha16)


# ------------------------------------------------------------------------------------------------ GPU: kernels
@gpu
@pytest.mark.parametrize("B", [0, 1, 3])
@pytest.mark.parametrize("H,W", KERNEL_SIZES)
def test_ingest_equals_torch(pkg, cuda_dev, B, H, W):
    for C in (4, 1):
        t = _random16(B, H, W, C, seed=H * 7 + W + B)
        image, alpha, size = pkg.rgba16_ingest(t.to(cuda_dev))
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
def test_ingest_covers_every_sample_value(pkg, cuda_dev):
    t = _random16(1, 256, 257, 4, seed=3)
    assert torch.equal(torch.unique(t[..., 3].to(torch.int32)), torch.arange(FULL + 1, dtype=torch.int32))
    image, alpha, _ = pkg.rgba16_ingest(t.to(cuda_dev))
    ref_image, ref_alpha = _ingest_ref(t)
    assert torch.equal(alpha.cpu(), ref_alpha) and torch.equal(image.cpu(), ref_image)
    # every value through the colour planes too: R = G = B = A
    t = _u16(t[..., 3:].to(torch.int32).repeat(1, 1, 1, 4))
    image, alpha, _ = pkg.rgba16_ingest(t.to(cuda_dev))
    ref_image, ref_alpha = _ingest_ref(t)
    assert torch.equal(image.cpu(), ref_image)


@gpu
def test_unaligned_inputs(pkg, lib, cuda_dev):
    """a buffer at an offset that breaks the 8-byte pixel alignment: the wrapper copies it, the ABI refuses it; alpha-only
    buffers and the egress' alpha need 2 bytes and run sample by sample; an RGBA output at 8 bytes runs pixel by pixel"""
    B, H, W = 2, 65, 63
    t = _random16(B, H, W, 4, seed=11)
    ref_image, ref_alpha = _ingest_ref(t)
    n = t.numel()
    buf = _zeros16(n + 4, cuda_dev)
    for k in (1, 2, 3):                                                # 2, 4, 6 bytes past an aligned allocation
        view = buf[k:k + n].view(B, H, W, 4)
        view.copy_(t.to(cuda_dev))
        image, alpha, _ = pkg.rgba16_ingest(view)
        assert torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha), k
        assert lib.rgba16_ingest(view.data_ptr(), image.data_ptr(), alpha.data_ptr(), B, H, W, 4,
                                 pkg._abi.stream_handle()) == -3
    a16 = t[..., 3].contiguous()
    _, ref_a = _ingest_ref(a16[..., None])
    abuf = _zeros16(a16.numel() + 1, cuda_dev)
    av = abuf[1:].view(B, H, W)
    av.copy_(a16.to(cuda_dev))
    alpha = torch.full((B, 1, _padded(H), _padded(W)), -1.0, device=cuda_dev)
    assert lib.rgba16_ingest(av.data_ptr(), None, alpha.data_ptr(), B, H, W, 1, pkg._abi.stream_handle()) == 0
    assert torch.equal(alpha.cpu(), ref_a)
    x = _specials(B, H, W, seed=12)
    xd = x.to(cuda_dev)
    want = _egress_ref(x, a16)
    out = _zeros16(B * H * W * 4 + 4, cuda_dev)
    assert lib.rgba16_egress(xd.data_ptr(), av.data_ptr(), out[4:].data_ptr(), B, H, W, pkg._abi.stream_handle()) == 0
    assert torch.equal(_i32(out[4:]).view(B, H, W, 4), want)
    assert lib.rgba16_egress(xd.data_ptr(), av.data_ptr(), out[2:].data_ptr(), B, H, W, pkg._abi.stream_handle()) == -3
    assert torch.equal(_i32(pkg.rgba16_egress(xd, av)), want)


@gpu
@pytest.mark.parametrize("B", [0, 1, 3])
@pytest.mark.parametrize("H,W", KERNEL_SIZES)
def test_egress_equals_torch(pkg, cuda_dev, B, H, W):
    x = _specials(B, H, W, seed=H + 3 * W + B)
    a16 = _random16(B, H, W, 1, seed=H + W + 11 * B)[..., 0].contiguous()
    got = pkg.rgba16_egress(x.to(cuda_dev), a16.to(cuda_dev))
    assert got.shape == (B, H, W, 4) and got.dtype == torch.uint16 and got.is_cuda
    assert torch.equal(_i32(got), _egress_ref(x, a16))


@gpu
@pytest.mark.parametrize("H,W", [(63, 65), (511, 767)])
def test_257_times_8_bit_gives_the_8_bit_planes(pkg, cuda_dev, H, W):
    t8 = torch.randint(0, 256, (2, H, W, 4), generator=torch.Generator().manual_seed(H), dtype=torch.uint8)
    t8.view(-1, 4)[:256, 3] = torch.arange(256, dtype=torch.uint8)              # every alpha value, none zeroed
    t16 = _times257(t8)
    i8, a8, _ = pkg.rgba8_ingest(t8.to(cuda_dev))
    i16, a16, _ = pkg.rgba16_ingest(t16.to(cuda_dev))
    assert torch.equal(i8, i16) and torch.equal(a8, a16)
    _, a8, _ = pkg.rgba8_ingest(t8[..., 3:].contiguous().to(cuda_dev))
    _, a16, _ = pkg.rgba16_ingest(t16[..., 3:].contiguous().to(cuda_dev))
    assert torch.equal(a8, a16)


@gpu
def test_host_inputs_side_stream_and_graph_capture(pkg, cuda_dev):
    B, H, W = 3, 63, 65
    t = _random16(B, H, W, 4, seed=5)
    x = _specials(B, H, W, seed=6)
    a16 = t[..., 3].contiguous()
    ref_image, ref_alpha = _ingest_ref(t)
    ref_out = _egress_ref(x, a16)
    # host inputs, pageable and pinned: copied to the device once
    for src in (t, t.pin_memory()):
        image, alpha, _ = pkg.rgba16_ingest(src)
        assert image.is_cuda and torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha)
    assert torch.equal(_i32(pkg.rgba16_egress(x.to(cuda_dev), a16.pin_memory())), ref_out)
    assert torch.equal(_i32(pkg.rgba16_egress(x.to(cuda_dev), a16)), ref_out)
    td, xd, ad = t.to(cuda_dev), x.to(cuda_dev), a16.to(cuda_dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        image, alpha, _ = pkg.rgba16_ingest(td)
        out = pkg.rgba16_egress(xd, ad)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha)
    assert torch.equal(_i32(out), ref_out)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        image, alpha, _ = pkg.rgba16_ingest(td)
        out = pkg.rgba16_egress(xd, ad)
    for _ in range(2):
        for o in (image, alpha):
            o.fill_(-1.0)
        out.view(torch.int16).fill_(7)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(image.cpu(), ref_image) and torch.equal(alpha.cpu(), ref_alpha)
        assert torch.equal(_i32(out), ref_out)


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
@pytest.mark.parametrize("H,W", [(63, 65), (192, 256)])
def test_257_times_8_bit_gives_the_8_bit_strings(cuda_dev, net, H, W):
    t8 = _image8(2, H, W, seed=H + W)
    t16 = _times257(t8)
    for coder in ("host", "device"):
        with torch.no_grad():
            a = net.compress_rgba8(t8.to(cuda_dev), coder=coder)
            b = net.compress_rgba16(t16.to(cuda_dev), coder=coder)
        assert b["size"] == a["size"] == (H, W) and tuple(b["shape"]) == tuple(a["shape"])
        assert a["strings"] == b["strings"], coder


@gpu
@pytest.mark.parametrize("H,W", [(63, 65), (511, 767)])
def test_round_trip_equals_torch_egress_of_decompress(pkg, cuda_dev, net, H, W):
    t = _image16(1, H, W, seed=2 * H + W)
    a16 = t[..., 3].contiguous()
    _, alpha, _ = pkg.rgba16_ingest(a16[..., None].to(cuda_dev))
    for coder, lanes in (("host", None), ("device", None), ("device", 7)):
        with torch.no_grad():
            out = net.compress_rgba16(t.to(cuda_dev), coder=coder, lanes=lanes)
            assert out["size"] == (H, W) and tuple(out["shape"]) == (_padded(H) // 64, _padded(W) // 64)
            rec = net.decompress_rgba16(out["strings"], out["shape"], a16.to(cuda_dev))
            x_hat = net.decompress(out["strings"], out["shape"], alpha)["x_hat"]
        assert rec.shape == (1, H, W, 4) and rec.dtype == torch.uint16
        rec = _i32(rec)
        assert torch.equal(rec, _egress_ref(x_hat.cpu(), a16)), (coder, lanes)
        assert torch.equal(rec[..., 3], a16.to(torch.int32))
        assert not rec[..., :3][a16.to(torch.int32) == 0].any()


@gpu
def test_8_bit_strings_decode_at_16_bits(pkg, cuda_dev, net):
    H, W = 63, 65
    t8 = _image8(1, H, W, seed=4)
    a8 = t8[..., 3].contiguous()
    a16 = _times257(a8)
    _, alpha, _ = pkg.rgba8_ingest(a8[..., None].to(cuda_dev))
    for coder in ("host", "device"):
        with torch.no_grad():
            out = net.compress_rgba8(t8.to(cuda_dev), coder=coder)
            rec = net.decompress_rgba16(out["strings"], out["shape"], a16)            # a host alpha: copied once
            x_hat = net.decompress(out["strings"], out["shape"], alpha)["x_hat"]
        assert torch.equal(_i32(rec), _egress_ref(x_hat.cpu(), a16)), coder


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
    t = _image16(2, 63, 65, seed=9)
    a16 = t[..., 3].contiguous().to(cuda_dev)
    t = t.to(cuda_dev)
    image, alpha, _ = pkg.rgba16_ingest(t)
    with torch.no_grad():
        for coder in ("host", "device"):                          # warm-up: tables on the device, kernels loaded
            out = net.compress_rgba16(t, coder=coder)
            net.compress(image, alpha, coder=coder)
            net.decompress_rgba16(out["strings"], out["shape"], a16)
        dev_out = net.compress_rgba16(t, coder="device")
        torch.cuda.synchronize()
        on_dev = _syncs(lambda: net.decompress_rgba16(dev_out["strings"], dev_out["shape"], a16))
        assert len(on_dev) <= 1, on_dev
        for coder in ("host", "device"):
            torch.cuda.synchronize()
            sixteen = _syncs(lambda: net.compress_rgba16(t, coder=coder))
            planes = _syncs(lambda: net.compress(image, alpha, coder=coder))
            assert len(sixteen) <= len(planes), (coder, sixteen, planes)
