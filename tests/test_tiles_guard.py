"""The size bounds around RGBA tiles (DESIGN.md 4.8), checked without a GPU: decompress_rgba8 / 16 keep the untiled
'too large' guard, decompress_tiled refuses a tile no forward pass can hold, and the tile entry points refuse a tile
grid whose rows or columns would leave int coordinates."""
import ctypes

import pytest
import torch


@pytest.mark.parametrize("dtype", [torch.uint8, torch.uint16])
@pytest.mark.parametrize("B,H,W", [(1, 8192, 8192), (114, 512, 768)])
def test_untiled_decompress_keeps_its_size_guard(pkg, dtype, B, H, W):
    net = pkg.RGBACodec().eval()
    alpha = torch.zeros(B, H, W, dtype=dtype)
    shape = (-(-H // 64), -(-W // 64))
    strings = [[b"\0" * 8] * B, [b"\0" * 8] * B]
    decompress = net.decompress_rgba8 if dtype == torch.uint8 else net.decompress_rgba16
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        decompress(strings, shape, alpha)
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        net.compress_rgba8(torch.zeros(B, H, W, 4, dtype=torch.uint8))


def test_tiled_decompress_refuses_a_tile_beyond_one_pass(pkg):
    net = pkg.RGBACodec().eval()
    alpha = torch.zeros(1, 8192, 8192, dtype=torch.uint8)
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        net.decompress_tiled([[b"\0" * 8], [b"\0" * 8]], (128, 128), alpha)
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        pkg.rgba8.tiles_of(8192, 8192, (128, 128))
    with pytest.raises(pkg.MwaB200Error, match="too large"):
        pkg.rgba8.chunk_tiles(8192, 8192)
    assert pkg.rgba8.tiles_of(8192, 8192, (64, 64)) == (4096, 4096, 2, 2)
    assert pkg.rgba8.tiles_of(64, 8192, (1, 128)) == (64, 8192, 1, 1)


@pytest.mark.parametrize("bits", [8, 16])
def test_tile_grid_stays_within_int_coordinates(lib, bits):
    """a tall (or wide) tile that passes the element bound but whose last tile row (column) would end at or past 2^31;
    the valid calls stop at a misaligned pointer, so nothing here launches"""
    odd = ctypes.c_void_p(257)
    ing, eg = getattr(lib, f"rgba{bits}_ingest_tiles"), getattr(lib, f"rgba{bits}_egress_tiles")
    big = 2 ** 31 - 1
    for H, W, Th, Tw in ((big, 1, 699008, 64), (1, big, 64, 699008)):
        assert ing(odd, odd, odd, 1, H, W, 4, Th, Tw, 0, 1, None) == -1, (H, W, Th, Tw)
        assert eg(odd, odd, odd, 1, H, W, Th, Tw, 0, 1, None) == -1, (H, W, Th, Tw)
    # tile rows that end below 2^31 are accepted: 3072 rows of 699008 end at 2,147,352,576
    assert ing(odd, odd, odd, 1, 2 ** 31 - 2 ** 17, 1, 4, 699008, 64, 3071, 1, None) == -3
    assert eg(odd, odd, odd, 1, 2 ** 31 - 2 ** 17, 1, 699008, 64, 3071, 1, None) == -3
