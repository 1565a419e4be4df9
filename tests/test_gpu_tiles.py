"""RGBA images in independent tiles (csrc/rgba8.cu's rgba{8,16}_ingest_tiles / _egress_tiles, <package>/rgba8.py's
tile_grid / ingest_tiles / egress_tiles, codec.AutoEncoder.compress_tiled / decompress_tiled; DESIGN.md 4.8).  The tile
geometry is checked exhaustively; the kernels are held bit for bit to torch expressions on the CPU (crop, zero-pad, IEEE
division, premultiply, quantise); every tile must be coded exactly as compress_rgba8 codes its crop padded by hand, and
decode exactly as decompress_rgba8 decodes that, however the tiles are chunked.  Argument checks run without a GPU."""
import ctypes
import os
import warnings

import pytest
import torch
import torch.nn.functional as F

from oracle import golden_cases as G

gpu = pytest.mark.gpu
FULL = {8: 255, 16: 65535}
DTYPE = {8: torch.uint8, 16: torch.uint16}


def _cdiv(a, b):
    return -(-a // b)


def _padded(n):
    return _cdiv(n, 64) * 64


def _as(t32, bits):
    """int32 samples as the uint8 / uint16 tensor (converted on the CPU, where both casts exist)"""
    return t32.cpu().to(DTYPE[bits])


def _i32(t):
    return t.cpu().to(torch.int32)


def _random(B, H, W, C, bits, seed):
    """uniform samples as int32, alpha zero on ~30 % of the pixels"""
    g = torch.Generator().manual_seed(seed)
    t = torch.randint(0, FULL[bits] + 1, (B, H, W, C), generator=g, dtype=torch.int32)
    t[..., -1] *= (torch.rand(B, H, W, generator=g) >= 0.3).to(torch.int32)
    return t


def _image8(B, H, W, seed):
    """uint8 (B, H, W, 4): smooth colour + noise, soft alpha with fully transparent 16 x 16 blocks, colour not premultiplied"""
    g = torch.Generator().manual_seed(seed)
    yy = torch.linspace(0, 1, H).view(1, H, 1)
    xx = torch.linspace(0, 1, W).view(1, 1, W)
    rgb = torch.stack([0.5 + 0.4 * torch.sin(6.0 * xx + 3.0 * yy), 0.5 + 0.4 * torch.cos(5.0 * yy - 2.0 * xx),
                       0.5 + 0.3 * torch.sin(9.0 * xx * yy + 1.0)], -1)
    rgb = (rgb + 0.08 * torch.randn(B, H, W, 3, generator=g)).clamp(0, 1)
    keep = torch.rand(B, _cdiv(H, 16), _cdiv(W, 16), generator=g) >= 0.35
    keep = keep.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :H, :W]
    alpha = (0.3 + 0.7 * torch.rand(B, H, W, generator=g)) * keep
    return (torch.cat([rgb, alpha[..., None]], -1) * 255).round().to(torch.uint8)


def _image16(B, H, W, seed):
    """the same kind of image at 16 bits, with values no 8-bit image has"""
    g = torch.Generator().manual_seed(seed + 1)
    t = _image8(B, H, W, seed).to(torch.int32) * 257 + torch.randint(-128, 129, (B, H, W, 4), generator=g, dtype=torch.int32)
    t = t.clamp(0, 65535)
    t[..., 3] *= (t[..., 3] > 200).to(torch.int32)
    return t.to(torch.uint16)


def _to_tiles(x, Th, Tw):
    """(B, C, ty * Th, tx * Tw) -> (B * ty * tx, C, Th, Tw) in tile order"""
    B, C, Hs, Ws = x.shape
    ty, tx = Hs // Th, Ws // Tw
    return x.view(B, C, ty, Th, tx, Tw).permute(0, 2, 4, 1, 3, 5).reshape(B * ty * tx, C, Th, Tw)


def _from_tiles(t, B, ty, tx):
    """_to_tiles inverted"""
    n, C, Th, Tw = t.shape
    return t.reshape(B, ty, tx, C, Th, Tw).permute(0, 3, 1, 4, 2, 5).reshape(B, C, ty * Th, tx * Tw)


def _ingest_ref(t32, bits, Th, Tw):
    """(image, alpha) of every tile: the int32 samples / full scale on the CPU (an IEEE division), zero-padded to the tile
    grid, colour premultiplied by the binarised alpha"""
    B, H, W, C = t32.shape
    f = F.pad(t32.permute(0, 3, 1, 2).float() / FULL[bits], (0, _cdiv(W, Tw) * Tw - W, 0, _cdiv(H, Th) * Th - H))
    alpha = f[:, C - 1:C]
    return (_to_tiles(f[:, :3] * (alpha > 0), Th, Tw) if C == 4 else None), _to_tiles(alpha, Th, Tw)


def _tile_index(B, H, W, Th, Tw):
    """(B, H, W): the tile each pixel belongs to"""
    b = torch.arange(B).view(B, 1, 1)
    i = (torch.arange(H) // Th).view(1, H, 1)
    j = (torch.arange(W) // Tw).view(1, 1, W)
    return (b * _cdiv(H, Th) + i) * _cdiv(W, Tw) + j


def _egress_ref(x_tiles, a32, bits, first, sentinel):
    """int32 (B, H, W, 4): where the pixel's tile is in [first, first + count), A = alpha and RGB = rint(clamp(x, 0, 1)
    * full) in fp32 where alpha > 0, else 0; elsewhere the sentinel"""
    count, _, Th, Tw = x_tiles.shape
    B, H, W = a32.shape
    ty, tx = _cdiv(H, Th), _cdiv(W, Tw)
    allt = torch.zeros(B * ty * tx, 3, Th, Tw)
    allt[first:first + count] = x_tiles
    x = _from_tiles(allt, B, ty, tx)[:, :, :H, :W]
    rgb = (x.nan_to_num(0).clamp(0, 1) * FULL[bits]).round().to(torch.int32) * (a32 > 0)[:, None]
    want = torch.cat([rgb.permute(0, 2, 3, 1), a32[..., None]], -1)
    n = _tile_index(B, H, W, Th, Tw)
    mine = ((n >= first) & (n < first + count))[..., None]
    return torch.where(mine, want, sentinel.to(torch.int32))


def _specials(n, Th, Tw, bits, seed):
    """fp32 (n, 3, Th, Tw) in [-0.5, 1.5] with NaN, +-Inf, exact 0 / 1 and k / full values sprinkled in"""
    g = torch.Generator().manual_seed(seed)
    x = torch.rand(n, 3, Th, Tw, generator=g) * 2 - 0.5
    pick = torch.rand(x.shape, generator=g)
    x[pick < 0.02] = float("nan")
    x[(pick >= 0.02) & (pick < 0.03)] = float("inf")
    x[(pick >= 0.03) & (pick < 0.04)] = float("-inf")
    x[(pick >= 0.04) & (pick < 0.05)] = 1.0
    x[(pick >= 0.05) & (pick < 0.06)] = 0.0
    k = (pick >= 0.06) & (pick < 0.1)
    x[k] = torch.randint(0, FULL[bits] + 1, (int(k.sum()),), generator=g).float() / FULL[bits]
    return x


def _sentinel(B, H, W, bits, device):
    """a (B, H, W, 4) output filled with 0x5a bytes, and the int32 value of that fill"""
    out = torch.full((B * H * W * 4 * bits // 8,), 0x5A, dtype=torch.uint8, device=device).view(DTYPE[bits])
    return out.view(B, H, W, 4), torch.tensor(0x5A5A if bits == 16 else 0x5A)


# ------------------------------------------------------------------------------------------------ CPU: the geometry
def test_tile_grid_exhaustive(pkg):
    """every Hp = 64 h, h < 160, every tile / 64 < 60, H at the top, middle and bottom of its 64-row band; the rule is per
    axis, so the width runs through the same cases transposed"""
    tile_grid = pkg.rgba8.tile_grid
    for h in range(1, 160):
        for H in {64 * h, 64 * h - 31, 64 * h - 63}:
            Hp = 64 * h
            for k in range(1, 60):
                tile = 64 * k
                Th, Tw, ty, tx = tile_grid(H, 64, tile)
                assert (Tw, tx) == (64, 1)
                assert Th % 64 == 0 and 64 <= Th <= tile, (H, tile, Th)
                assert ty * Th >= Hp, (H, tile)                           # the tiles cover the image
                assert (ty - 1) * Th < H, (H, tile)                       # no tile lies wholly outside it
                assert ty == _cdiv(H, Th) == _cdiv(Hp, tile), (H, tile)
                assert ty * Th - Hp < 64 * ty, (H, tile)                  # under 64 rows of padding per tile row
                if tile >= Hp:
                    assert (Th, ty) == (Hp, 1)
                assert tile_grid(64, H, tile) == (64, Th, 1, ty)
                assert pkg.rgba8.tiles_of(H, 64, (Th // 64, 1)) == (Th, 64, ty, 1)
    assert tile_grid(8192, 8192, 4096) == (4096, 4096, 2, 2)
    assert tile_grid(9001, 7003, 4096) == (3008, 3520, 3, 2)
    assert tile_grid(200, 330, 128) == (128, 128, 2, 3)
    assert tile_grid(200, 330, 192) == (128, 192, 2, 2)
    assert tile_grid(512, 768, 4096) == (512, 768, 1, 1)
    assert tile_grid(1, 1, 6656) == (64, 64, 1, 1)
    for bad in (0, 32, 100, -64, 6720, 8192, 64.0, "64", True, None):
        with pytest.raises(ValueError, match="tile"):
            tile_grid(100, 100, bad)


def test_shape_must_fit_the_alpha(pkg):
    tiles_of = pkg.rgba8.tiles_of
    assert tiles_of(200, 330, (2, 3)) == (128, 192, 2, 2)
    assert tiles_of(200, 330, (4, 6)) == (256, 384, 1, 1)                  # untiled
    assert tiles_of(64, 8192, (1, 128)) == (64, 8192, 1, 1)                # untiled, wider than any tile
    for shape in ((5, 1), (3, 3), (4, 5), (2, 7), (0, 2), (-1, 2), (2,), (2, 3, 1), "ab", None):
        with pytest.raises(ValueError, match="shape"):
            tiles_of(200, 330, shape)


# ------------------------------------------------------------------------------------------------ CPU: arguments
@pytest.mark.parametrize("bits", [8, 16])
def test_status_codes_before_any_launch(lib, bits):
    """calls that pass every size check are stopped at a misaligned pointer: nothing here launches"""
    one, odd = ctypes.c_void_p(256), ctypes.c_void_p(257)
    ing, eg = getattr(lib, f"rgba{bits}_ingest_tiles"), getattr(lib, f"rgba{bits}_egress_tiles")

    def both(B, H, W, Th, Tw, first, count, ptrs=(one, one, one)):
        return ing(*ptrs, B, H, W, 4, Th, Tw, first, count, None), eg(*ptrs, B, H, W, Th, Tw, first, count, None)

    # null pointers
    assert ing(None, one, one, 1, 100, 100, 4, 64, 64, 0, 4, None) == -1
    assert ing(one, None, one, 1, 100, 100, 4, 64, 64, 0, 4, None) == -1
    assert ing(one, one, None, 1, 100, 100, 4, 64, 64, 0, 4, None) == -1
    assert ing(None, None, one, 1, 100, 100, 1, 64, 64, 0, 4, None) == -1
    assert eg(None, one, one, 1, 100, 100, 64, 64, 0, 4, None) == -1
    assert eg(one, None, one, 1, 100, 100, 64, 64, 0, 4, None) == -1
    assert eg(one, one, None, 1, 100, 100, 64, 64, 0, 4, None) == -1
    # sizes, channels and tile sides
    for B, H, W in ((-1, 8, 8), (1, 0, 8), (1, 8, 0), (1, -5, 8)):
        assert both(B, H, W, 64, 64, 0, 1) == (-1, -1), (B, H, W)
    for C in (0, 2, 3, 5, -4):
        assert ing(one, one, one, 1, 8, 8, C, 64, 64, 0, 1, None) == -1, C
    for Th, Tw in ((0, 64), (64, 0), (32, 64), (64, 96), (-64, 64), (100, 64)):
        assert both(1, 100, 100, Th, Tw, 0, 1) == (-1, -1), (Th, Tw)
    # ranges: 2 images of 100 x 100 in tiles of 64 x 64 are 2 * 2 * 2 = 8 tiles
    assert both(2, 100, 100, 64, 64, 0, 8, (odd, odd, odd)) == (-3, -3)
    assert both(2, 100, 100, 64, 64, 7, 1, (odd, odd, odd)) == (-3, -3)
    assert both(2, 100, 100, 64, 64, 0, 9) == (-1, -1)
    assert both(2, 100, 100, 64, 64, 8, 1) == (-1, -1)
    assert both(2, 100, 100, 64, 64, -1, 1) == (-1, -1)
    assert both(2, 100, 100, 64, 64, 0, -1) == (-1, -1)
    assert both(2, 100, 100, 64, 64, 9, 0) == (-1, -1)
    assert both(2, 100, 100, 64, 64, 2 ** 63 - 1, 1) == (-1, -1)         # first + count overflows int64
    assert both(2 ** 31 - 1, 2 ** 31 - 1, 2 ** 31 - 1, 64, 64, 2 ** 62, 0) == (0, 0)      # in range, nothing to do
    # count * Th * Tw * 48 < 2^31: two tiles of 4096 x 4096 (an 8192 x 8192 image), not three; one of 6656 x 6656
    assert both(1, 8192, 8192, 4096, 4096, 0, 2, (odd, odd, odd)) == (-3, -3)
    assert both(1, 8192, 8192, 4096, 4096, 1, 3) == (-1, -1)
    assert both(1, 6656, 6656, 6656, 6656, 0, 1, (odd, odd, odd)) == (-3, -3)
    assert both(1, 6720, 6720, 6720, 6720, 0, 1) == (-1, -1)
    assert both(1, 64, 2 ** 31 - 64, 64, 2 ** 31 - 64, 0, 1) == (-1, -1)
    # the images themselves may exceed 2^31 bytes
    assert both(3, 20000, 20000, 4096, 4096, 74, 1, (odd, odd, odd)) == (-3, -3)
    # alignment: the rules of the untiled entry points
    word = 4 if bits == 8 else 8
    mis = ctypes.c_void_p(256 + word // 2)
    assert ing(one, one, odd, 1, 100, 100, 4, 64, 64, 0, 1, None) == -3
    assert ing(one, odd, one, 1, 100, 100, 4, 64, 64, 0, 1, None) == -3
    assert ing(mis, one, one, 1, 100, 100, 4, 64, 64, 0, 1, None) == -3
    assert eg(odd, one, one, 1, 100, 100, 64, 64, 0, 1, None) == -3
    assert eg(one, one, mis, 1, 100, 100, 64, 64, 0, 1, None) == -3
    if bits == 16:
        assert ing(odd, None, one, 1, 100, 100, 1, 64, 64, 0, 1, None) == -3
        assert eg(one, odd, one, 1, 100, 100, 64, 64, 0, 1, None) == -3
    # count = 0 launches nothing, whatever the pointers
    assert ing(None, None, None, 1, 100, 100, 4, 64, 64, 0, 0, None) == 0
    assert ing(None, None, None, 1, 100, 100, 1, 64, 64, 4, 0, None) == 0
    assert eg(None, None, None, 1, 100, 100, 64, 64, 2, 0, None) == 0
    assert eg(odd, odd, odd, 0, 100, 100, 64, 64, 0, 0, None) == 0


def test_python_wrappers_reject_bad_inputs(pkg):
    r = pkg.rgba8
    good = torch.zeros(2, 100, 100, 4, dtype=torch.uint8)
    for bad in (good.float(), good.to(torch.int32), good.to(torch.int16)):
        with pytest.raises(pkg.MwaB200Error, match="uint8 or uint16"):
            r.ingest_tiles(bad, (64, 64), 0, 1)
    with pytest.raises(ValueError):
        r.ingest_tiles(good.numpy(), (64, 64), 0, 1)
    for shape in ((100, 100), (2, 100, 100, 3), (1, 2, 100, 100, 4)):
        with pytest.raises(ValueError):
            r.ingest_tiles(torch.zeros(shape, dtype=torch.uint16), (64, 64), 0, 1)
    with pytest.raises(ValueError, match="contiguous"):
        r.ingest_tiles(good.transpose(1, 2), (64, 64), 0, 1)
    for tile_hw in ((0, 64), (64, 96), (32, 32)):
        with pytest.raises(ValueError, match="multiples of 64"):
            r.ingest_tiles(good, tile_hw, 0, 1)
    for first, count in ((-1, 1), (0, -1), (0, 9), (8, 1)):
        with pytest.raises(ValueError, match="not within"):
            r.ingest_tiles(good, (64, 64), first, count)
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        r.ingest_tiles(torch.zeros(1, 8192, 8192, 1, dtype=torch.uint8), (4096, 4096), 0, 3)
    with pytest.raises(pkg.MwaB200Error, match="CUDA"):
        r.egress_tiles(torch.zeros(1, 3, 64, 64), torch.zeros(1, 5, 7, dtype=torch.uint8),
                       torch.zeros(1, 5, 7, 4, dtype=torch.uint8), 0)


def test_codec_rejects_bad_arguments_before_any_launch(pkg):
    net = pkg.RGBACodec().eval()
    img = torch.zeros(200, 330, 4, dtype=torch.uint8)
    with pytest.raises(ValueError, match="coder"):
        net.compress_tiled(img, 128, coder="gpu")
    for bad in (img.float(), img.to(torch.int32)):
        with pytest.raises(pkg.MwaB200Error, match="uint8 or uint16"):
            net.compress_tiled(bad, 128)
    with pytest.raises(ValueError):
        net.compress_tiled(img[..., :1].contiguous(), 128)                # alpha alone is not an image
    with pytest.raises(ValueError, match="contiguous"):
        net.compress_tiled(torch.zeros(330, 200, 4, dtype=torch.uint8).transpose(0, 1), 128)
    for tile in (100, 32, 6720):
        with pytest.raises(ValueError, match="tile"):
            net.compress_tiled(img, tile)
    alpha = torch.zeros(2, 200, 330, dtype=torch.uint16)
    s6 = [b"\0" * 8] * 6
    for shape in ((5, 1), (3, 3), (4, 5), (2,)):                       # no tile grid of 200 x 330 has these tiles
        with pytest.raises(ValueError, match="shape"):
            net.decompress_tiled([s6 * 2, s6 * 2], shape, alpha)
    for strings in ([s6, s6 * 2], [s6 * 2, s6], [s6 * 2], [s6 * 2, s6 * 2, s6 * 2]):   # 2 images of 2 x 3 tiles: 12
        with pytest.raises(ValueError, match="12 tiles"):
            net.decompress_tiled(strings, (2, 2), alpha)
    with pytest.raises(ValueError, match="2 tiles"):
        net.decompress_tiled([s6, s6], (4, 6), alpha)                    # untiled: one tile per image
    with pytest.raises(pkg.MwaB200Error, match="uint8 or uint16"):
        net.decompress_tiled([s6 * 2, s6 * 2], (2, 2), alpha.to(torch.int32))
    with pytest.raises(ValueError, match="contiguous"):
        net.decompress_tiled([s6, s6], (2, 2), torch.zeros(330, 200, dtype=torch.uint8).t())


# ------------------------------------------------------------------------------------------------ GPU: kernels
@gpu
@pytest.mark.parametrize("bits", [8, 16])
@pytest.mark.parametrize("B,H,W,Th,Tw", [(1, 1, 1, 64, 64), (2, 63, 130, 64, 64), (3, 129, 67, 128, 64),
                                         (2, 200, 330, 128, 192), (1, 257, 255, 320, 256)])
def test_tile_kernels_equal_torch(pkg, cuda_dev, bits, B, H, W, Th, Tw):
    r = pkg.rgba8
    n = B * _cdiv(H, Th) * _cdiv(W, Tw)
    ranges = {(0, n), (0, 1), (n - 1, 1), (n // 2, n - n // 2), (1, max(n - 2, 0))}
    for C in (4, 1):
        t32 = _random(B, H, W, C, bits, seed=H + W + C + bits)
        td = _as(t32, bits).to(cuda_dev)
        ref_image, ref_alpha = _ingest_ref(t32, bits, Th, Tw)
        for first, count in sorted(ranges):
            image, alpha = r.ingest_tiles(td, (Th, Tw), first, count)
            assert alpha.shape == (count, 1, Th, Tw) and alpha.dtype == torch.float32
            assert torch.equal(alpha.cpu(), ref_alpha[first:first + count]) and not torch.signbit(alpha).any()
            if C == 4:
                assert image.shape == (count, 3, Th, Tw)
                assert torch.equal(image.cpu(), ref_image[first:first + count]) and not torch.signbit(image).any()
            else:
                assert image is None
    a32 = t32[..., 0]
    ad = _as(a32, bits).to(cuda_dev)
    for first, count in sorted(ranges):
        x = _specials(count, Th, Tw, bits, seed=first + 7 * count)
        out, sentinel = _sentinel(B, H, W, bits, cuda_dev)
        assert r.egress_tiles(x.to(cuda_dev), ad, out, first) is out
        assert torch.equal(_i32(out), _egress_ref(x, a32, bits, first, sentinel)), (first, count)


@gpu
@pytest.mark.parametrize("bits", [8, 16])
def test_untiled_entry_points_are_the_one_tile_case(pkg, cuda_dev, bits):
    """rgba*_ingest / _egress give exactly the planes and pixels of one Hp x Wp tile per image"""
    B, H, W = 3, 65, 127
    t32 = _random(B, H, W, 4, bits, seed=bits)
    td = _as(t32, bits).to(cuda_dev)
    image, alpha, _ = getattr(pkg, f"rgba{bits}_ingest")(td)
    ti, ta = pkg.rgba8.ingest_tiles(td, (_padded(H), _padded(W)), 0, B)
    assert torch.equal(image, ti) and torch.equal(alpha, ta)
    x = _specials(B, _padded(H), _padded(W), bits, seed=3).to(cuda_dev)
    ad = td[..., 3].contiguous()
    out, _ = _sentinel(B, H, W, bits, cuda_dev)
    pkg.rgba8.egress_tiles(x, ad, out, 0)
    assert torch.equal(_i32(out), _i32(getattr(pkg, f"rgba{bits}_egress")(x, ad)))


@gpu
@pytest.mark.parametrize("bits", [8, 16])
def test_unaligned_views_side_stream_and_graph_replay(pkg, lib, cuda_dev, bits):
    r = pkg.rgba8
    B, H, W, Th, Tw = 2, 130, 70, 64, 64                                    # 3 x 2 tiles per image
    first, count = 2, 7
    t32 = _random(B, H, W, 4, bits, seed=21)
    ref_image, ref_alpha = _ingest_ref(t32, bits, Th, Tw)
    want_i, want_a = ref_image[first:first + count], ref_alpha[first:first + count]
    n = t32.numel()
    buf = torch.zeros(n + 4, dtype=DTYPE[bits], device=cuda_dev)
    for k in (1, 2, 3):                                                    # off the 4-sample Word boundary
        view = buf[k:k + n].view(B, H, W, 4)
        view.copy_(_as(t32, bits).to(cuda_dev))
        image, alpha = r.ingest_tiles(view, (Th, Tw), first, count)       # the wrapper copies it once
        assert torch.equal(image.cpu(), want_i) and torch.equal(alpha.cpu(), want_a), k
        assert getattr(lib, f"rgba{bits}_ingest_tiles")(view.data_ptr(), image.data_ptr(), alpha.data_ptr(), B, H, W,
                                                        4, Th, Tw, first, count, pkg._abi.stream_handle()) == -3
    # an alpha at an odd sample offset and an RGBA output at a Word but not 16-byte boundary: sample by sample
    a32 = t32[..., 3].contiguous()
    abuf = torch.zeros(a32.numel() + 1, dtype=DTYPE[bits], device=cuda_dev)
    av = abuf[1:].view(B, H, W)
    av.copy_(_as(a32, bits).to(cuda_dev))
    _, alpha = r.ingest_tiles(av[..., None], (Th, Tw), first, count)
    assert torch.equal(alpha.cpu(), want_a)
    x = _specials(count, Th, Tw, bits, seed=22)
    xd = x.to(cuda_dev)
    obuf = torch.full((B * H * W * 4 + 4,), 0x5A5A if bits == 16 else 0x5A, dtype=torch.int32).to(DTYPE[bits]).to(cuda_dev)
    out = obuf[4:].view(B, H, W, 4)
    sentinel = torch.tensor(0x5A5A if bits == 16 else 0x5A)
    want = _egress_ref(x, a32, bits, first, sentinel)
    r.egress_tiles(xd, av, out, first)
    assert torch.equal(_i32(out), want)
    assert torch.equal(_i32(obuf[:4]), sentinel.expand(4).to(torch.int32))
    # a side stream, then graph replay
    td, ad = _as(t32, bits).to(cuda_dev), _as(a32, bits).to(cuda_dev)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    out, _ = _sentinel(B, H, W, bits, cuda_dev)
    with torch.cuda.stream(side):
        image, alpha = r.ingest_tiles(td, (Th, Tw), first, count)
        r.egress_tiles(xd, ad, out, first)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(image.cpu(), want_i) and torch.equal(alpha.cpu(), want_a)
    assert torch.equal(_i32(out), want)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        image, alpha = r.ingest_tiles(td, (Th, Tw), first, count)
        r.egress_tiles(xd, ad, out, first)
    for _ in range(2):
        image.fill_(-1.0), alpha.fill_(-1.0)
        out.view(torch.uint8).fill_(0x5A)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(image.cpu(), want_i) and torch.equal(alpha.cpu(), want_a)
        assert torch.equal(_i32(out), want)


@gpu
def test_egress_rejects_bad_arguments_before_any_launch(pkg, cuda_dev):
    r = pkg.rgba8
    x = torch.zeros(2, 3, 64, 64, device=cuda_dev)
    a8 = torch.zeros(1, 100, 100, dtype=torch.uint8, device=cuda_dev)
    out8 = torch.zeros(1, 100, 100, 4, dtype=torch.uint8, device=cuda_dev)
    launches = pkg._abi.launch_count
    with pytest.raises(pkg.MwaB200Error, match="uint8 or uint16"):
        r.egress_tiles(x, a8.float(), out8, 0)
    with pytest.raises(ValueError, match="out"):
        r.egress_tiles(x, a8, out8.to(torch.int16).view(torch.uint16), 0)           # dtype of the alpha
    for bad in (out8[:, :99], out8.cpu(), out8.transpose(1, 2), out8[..., :3]):
        with pytest.raises(ValueError, match="out"):
            r.egress_tiles(x, a8, bad, 0)
    with pytest.raises(ValueError, match="alpha8"):
        r.egress_tiles(x, a8[0], out8, 0)
    with pytest.raises(ValueError, match="x_hat"):
        r.egress_tiles(x[:, :2], a8, out8, 0)
    with pytest.raises(ValueError, match="multiples of 64"):
        r.egress_tiles(torch.zeros(2, 3, 64, 96, device=cuda_dev), a8, out8, 0)
    with pytest.raises(ValueError, match="not within"):
        r.egress_tiles(x, a8, out8, 3)                                   # 4 tiles of 64 x 64: [3, 5) is not
    assert pkg._abi.launch_count == launches


# ------------------------------------------------------------------------------------------------ GPU: the codec
@pytest.fixture
def net(pkg, cuda_dev, model_keys):
    """the codec on G.model_state weights, cuDNN held to deterministic algorithms: the comparisons below are exact"""
    prev = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    model = pkg.RGBACodec().eval()
    model.load_state_dict(G.model_state(model_keys, 61), strict=False)
    try:
        yield model.to(cuda_dev)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev


def _signed(t):
    """a uint16 tensor as int16, the same bits: torch has few CUDA kernels for uint16"""
    return t.view(torch.int16) if t.dtype == torch.uint16 else t


def _alpha(t):
    """the alpha channel of (B, H, W, 4), contiguous"""
    return _signed(t)[..., 3].contiguous().view(t.dtype)


def _crops(t, Th, Tw, tiles):
    """(count, Th, Tw, C): the crops of tiles [tiles[0], tiles[1]) of t (B, H, W, C), zero-padded by hand (zero alpha:
    transparent)"""
    B, H, W, C = t.shape
    ty, tx = _cdiv(H, Th), _cdiv(W, Tw)
    s = _signed(t)
    p = torch.zeros(B, ty * Th, tx * Tw, C, dtype=s.dtype, device=t.device)
    p[:, :H, :W] = s
    c = p.view(B, ty, Th, tx, Tw, C).permute(0, 1, 3, 2, 4, 5).reshape(B * ty * tx, Th, Tw, C)
    return c[tiles[0]:tiles[1]].contiguous().view(t.dtype)


def _stitch(crops, B, H, W):
    """the list of (count, Th, Tw, C) crops of _crops, in tile order, stitched and cropped to (B, H, W, C)"""
    c = torch.cat([_signed(k) for k in crops])
    n, Th, Tw, C = c.shape
    ty, tx = _cdiv(H, Th), _cdiv(W, Tw)
    c = c.view(B, ty, tx, Th, Tw, C).permute(0, 1, 3, 2, 4, 5).reshape(B, ty * Th, tx * Tw, C)[:, :H, :W]
    return c.contiguous().view(crops[0].dtype)


def _per_tile(net, t, Th, Tw, per, coder):
    """compress_rgba8 / 16 of the tiles' crops and decompress_rgba8 / 16 of their strings, stitched, in passes of `per`
    tiles (the passes compress_tiled makes): (strings, decoded (B, H, W, 4))"""
    B, H, W, _ = t.shape
    bits = 8 * t.element_size()
    n = B * _cdiv(H, Th) * _cdiv(W, Tw)
    strings, rec = [[], []], []
    for first in range(0, n, per):
        c = _crops(t, Th, Tw, (first, min(first + per, n)))
        out = getattr(net, f"compress_rgba{bits}")(c, coder=coder)
        rec.append(getattr(net, f"decompress_rgba{bits}")(out["strings"], out["shape"], _alpha(c)))
        strings[0] += out["strings"][0]
        strings[1] += out["strings"][1]
    return strings, _stitch(rec, B, H, W)


@gpu
@pytest.mark.parametrize("tile,grid,shape", [(128, (2, 3), (2, 2)), (192, (2, 2), (2, 3))])
def test_tiles_are_coded_as_their_padded_crops(pkg, cuda_dev, net, tile, grid, shape):
    t = _image8(2, 200, 330, seed=tile).to(cuda_dev)
    a8 = t[..., 3].contiguous()
    for coder in ("host", "device"):
        with torch.no_grad():
            out = net.compress_tiled(t, tile, coder=coder)
            assert out["grid"] == grid and tuple(out["shape"]) == shape and out["size"] == (200, 330)
            assert len(out["strings"][0]) == len(out["strings"][1]) == 2 * grid[0] * grid[1]
            strings, want = _per_tile(net, t, 64 * shape[0], 64 * shape[1], 2 * grid[0] * grid[1], coder)
            assert out["strings"] == strings, coder
            rec = net.decompress_tiled(out["strings"], out["shape"], a8)
        assert rec.shape == (2, 200, 330, 4) and rec.dtype == torch.uint8
        assert torch.equal(rec, want), coder
        assert torch.equal(rec[..., 3], a8) and not rec[..., :3][a8 == 0].any()


@gpu
def test_one_tile_is_the_untiled_path(pkg, cuda_dev, net):
    t = _image8(2, 200, 330, seed=5).to(cuda_dev)
    a8 = t[..., 3].contiguous()
    for coder in ("host", "device"):
        with torch.no_grad():
            ref = net.compress_rgba8(t, coder=coder)
            for tile in (384, 6656):
                out = net.compress_tiled(t, tile, coder=coder)
                assert out["grid"] == (1, 1) and tuple(out["shape"]) == tuple(ref["shape"]) == (4, 6)
                assert out["strings"] == ref["strings"], (coder, tile)
            rec = net.decompress_rgba8(ref["strings"], ref["shape"], a8)
            assert torch.equal(net.decompress_tiled(ref["strings"], ref["shape"], a8), rec)
            assert torch.equal(net.decompress_rgba8(out["strings"], out["shape"], a8), rec)


@gpu
def test_16_bit_tiles(pkg, cuda_dev, net):
    """257 * v gives v's strings; a 16-bit round trip equals the 16-bit decode of the padded crops"""
    t8 = _image8(2, 200, 330, seed=8)
    t16 = (t8.to(torch.int32) * 257).to(torch.uint16)
    for coder in ("host", "device"):
        with torch.no_grad():
            a = net.compress_tiled(t8.to(cuda_dev), 128, coder=coder)
            b = net.compress_tiled(t16.to(cuda_dev), 128, coder=coder)
            assert a["strings"] == b["strings"] and a["grid"] == b["grid"] and tuple(a["shape"]) == tuple(b["shape"])
    t = _image16(1, 200, 330, seed=9)
    with torch.no_grad():
        out = net.compress_tiled(t, 192, coder="device")                  # a host input: copied once
        strings, want = _per_tile(net, t.to(cuda_dev), 128, 192, 4, "device")
        assert out["strings"] == strings
        rec = net.decompress_tiled(out["strings"], out["shape"], _alpha(t))
    assert rec.dtype == torch.uint16 and torch.equal(_i32(rec), _i32(want))


@gpu
@pytest.mark.parametrize("per", [1, 2, 3, 5])
def test_chunking_does_not_change_the_result(pkg, cuda_dev, net, monkeypatch, per):
    """passes of 1, 2, 3 or 5 of the 12 tiles (boundaries inside an image) give the strings and pixels of one pass"""
    t = _image8(2, 200, 330, seed=13).to(cuda_dev)
    a8 = t[..., 3].contiguous()
    with torch.no_grad():
        ref = {c: net.compress_tiled(t, 128, coder=c) for c in ("host", "device")}
        rec = net.decompress_tiled(ref["device"]["strings"], ref["device"]["shape"], a8)
        monkeypatch.setattr(pkg.rgba8, "MAX_ELEMENTS", per * 128 * 128 * 48 + 1)
        assert pkg.rgba8.chunk_tiles(128, 128) == per
        for coder in ("host", "device"):
            out = net.compress_tiled(t, 128, coder=coder)
            assert out["strings"] == ref[coder]["strings"], (per, coder)
            assert torch.equal(net.decompress_tiled(out["strings"], out["shape"], a8), rec), (per, coder)


@gpu
@pytest.mark.parametrize("bits,H,W", [(8, 8192, 8192), (16, 9001, 7003)])
def test_large_images(pkg, cuda_dev, net, bits, H, W):
    """beyond one pass: at the default tile each round trip equals the per-tile coding of the padded crops"""
    g = torch.Generator(device=cuda_dev).manual_seed(bits)
    small = _image8(1, _cdiv(H, 16), _cdiv(W, 16), seed=bits).to(cuda_dev)
    t = small.repeat_interleave(16, 1).repeat_interleave(16, 2)[:, :H, :W].to(torch.int32)
    if bits == 16:
        t = t * 257 + torch.randint(-100, 101, t.shape, generator=g, device=cuda_dev, dtype=torch.int32)
        t[..., 3] *= (t[..., 3] > 300).to(torch.int32)
        t = t.clamp(0, 65535).to(torch.int32)
    t = t.to(DTYPE[bits]) if bits == 8 else t.cpu().to(torch.uint16).to(cuda_dev)
    alpha = _alpha(t)
    Th, Tw, ty, tx = pkg.rgba8.tile_grid(H, W, 4096)
    if bits == 8:
        with pytest.raises(pkg.MwaB200Error, match="too large"):
            net.compress_rgba8(t)
    for coder in ("host", "device"):
        with torch.no_grad():
            out = net.compress_tiled(t, coder=coder)
            assert out["grid"] == (ty, tx) and tuple(out["shape"]) == (Th // 64, Tw // 64)
            strings, want = _per_tile(net, t, Th, Tw, pkg.rgba8.chunk_tiles(Th, Tw), coder)
            assert out["strings"] == strings, coder
            del strings
            rec = net.decompress_tiled(out["strings"], out["shape"], alpha)
        assert rec.shape == (1, H, W, 4) and torch.equal(rec.view(torch.uint8), want.view(torch.uint8)), coder
        del rec, want


@gpu
def test_a_batch_beyond_one_pass(pkg, cuda_dev, net):
    """200 images of 768 x 512: one tile each, in passes of 113 and 87"""
    t = _image8(8, 512, 768, seed=17).repeat(25, 1, 1, 1).to(cuda_dev)
    t[:, 0, 0, :] = torch.arange(200, device=cuda_dev, dtype=torch.uint8)[:, None]      # no two images alike
    a8 = t[..., 3].contiguous()
    assert pkg.rgba8.chunk_tiles(512, 768) == 113
    with torch.no_grad():
        out = net.compress_tiled(t, coder="device")
        assert out["grid"] == (1, 1) and tuple(out["shape"]) == (8, 12) and len(out["strings"][0]) == 200
        rec = net.decompress_tiled(out["strings"], out["shape"], a8)
        tail = net.decompress_rgba8([s[113:] for s in out["strings"]], out["shape"], a8[113:])
        assert [s[113:] for s in out["strings"]] == net.compress_rgba8(t[113:], coder="device")["strings"]
    assert torch.equal(rec[113:], tail)
    assert torch.equal(rec[..., 3], a8) and not rec[..., :3][a8 == 0].any()


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
def test_synchronisation_counts(pkg, cuda_dev, net, monkeypatch):
    t = _image8(2, 200, 330, seed=19).to(cuda_dev)
    a8 = t[..., 3].contiguous()
    monkeypatch.setattr(pkg.rgba8, "MAX_ELEMENTS", 5 * 128 * 128 * 48 + 1)         # 12 tiles in 3 passes
    chunks = 3
    with torch.no_grad():
        image, alpha = pkg.rgba8.ingest_tiles(t, (128, 128), 0, 5)
        for coder in ("host", "device"):                                 # warm-up
            out = net.compress_tiled(t, 128, coder=coder)
            net.compress(image, alpha, coder=coder)
            net.decompress_tiled(out["strings"], out["shape"], a8)
        torch.cuda.synchronize()
        on_dev = _syncs(lambda: net.decompress_tiled(out["strings"], out["shape"], a8))
        assert len(on_dev) <= chunks, on_dev
        for coder in ("host", "device"):
            torch.cuda.synchronize()
            tiled = _syncs(lambda: net.compress_tiled(t, 128, coder=coder))
            planes = _syncs(lambda: net.compress(image, alpha, coder=coder))
            assert len(tiled) <= chunks * len(planes), (coder, tiled, planes)
