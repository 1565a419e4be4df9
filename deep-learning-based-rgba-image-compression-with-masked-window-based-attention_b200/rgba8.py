"""8- and 16-bit RGBA images of any size in and out of the codec (csrc/rgba8.cu, DESIGN.md 4.8).

    rgba8_ingest(rgba8)            uint8 (B, H, W, 4) or (H, W, 4) -> fp32 image (B, 3, Hp, Wp), alpha (B, 1, Hp, Wp), (H, W)
                                   uint8 (..., 1) (alpha only)     -> None, alpha, (H, W)
    rgba8_egress(x_hat, alpha8)    fp32 (B, 3, Hp, Wp) + uint8 (B, H, W) -> uint8 (B, H, W, 4) on x_hat's device
    rgba16_ingest / rgba16_egress  the same for uint16 samples, full scale 65535

    tile_grid(H, W, tile)                           -> (Th, Tw, ty, tx): the tiles of an image too large for one pass
    ingest_tiles(t, (Th, Tw), first, count)         uint8 / uint16 (B, H, W, C) -> the planes of tiles [first, first + count)
    egress_tiles(x_hat, alpha, out, first)          fp32 (count, 3, Th, Tw) -> the pixels of `out` (B, H, W, 4) they cover

Hp / Wp are H / W rounded up to a multiple of 64 (the model's coarsest stride: z is Hp / 64 x Wp / 64); the padding, at the
bottom and right, is transparent.  The planes are what the model was trained on: a / full scale and the colour
premultiplied by the binarised alpha.  One kernel launch each way.
"""
from __future__ import annotations

import torch

from . import _abi

PAD = 64
# B * Hp * Wp * 48 (the forward's largest activation, 192 channels at 1/2 scale) must stay below 2^31: the C entry points'
# guard, checked here too so that the planes are not allocated for an input they will refuse
MAX_ELEMENTS = 2 ** 31


def padded(n: int) -> int:
    return -(-n // PAD) * PAD


def tile_grid(H: int, W: int, tile: int):
    """(Th, Tw, ty, tx): the tiles of an H x W image for a requested `tile` (a multiple of 64, 64 <= tile, tile^2 * 48 <
    2^31).  The padded image splits into ty = ceil(Hp / tile) rows and tx = ceil(Wp / tile) columns of equal tiles,
    Th = 64 * ceil(Hp / (64 * ty)) <= tile (and Tw alike), so the padding stays under 64 rows per tile row instead of up
    to a whole tile.  ty = ceil(H / Th) and tx = ceil(W / Tw): the decoder recovers the grid from (H, W) and (Th, Tw).
    tile >= max(Hp, Wp) gives one Hp x Wp tile, the untiled geometry."""
    if isinstance(tile, bool) or not isinstance(tile, int) or tile < PAD or tile % PAD or tile * tile * 48 >= 2 ** 31:
        raise ValueError(f"tile must be a multiple of {PAD} from {PAD} to 6656 (tile^2 * 48 < 2^31; got {tile!r})")
    if H < 1 or W < 1:
        raise ValueError(f"image height and width must be >= 1 (got {H} x {W})")
    Hp, Wp = padded(H), padded(W)
    ty, tx = -(-Hp // tile), -(-Wp // tile)
    return padded(-(-Hp // ty)), padded(-(-Wp // tx)), ty, tx


def tiles_of(H: int, W: int, shape):
    """(Th, Tw, ty, tx) of the tiles whose z is `shape` = (Th / 64, Tw / 64) in an H x W image: the grid is (ceil(H / Th),
    ceil(W / Tw)), and the shape must be the one tile_grid gives for it (or the untiled Hp x Wp).  ValueError otherwise."""
    try:
        Th, Tw = (int(v) * PAD for v in shape)
    except (TypeError, ValueError):
        raise ValueError(f"shape must be (Th / {PAD}, Tw / {PAD}) (got {shape!r})") from None
    if Th < PAD or Tw < PAD:
        raise ValueError(f"shape {tuple(shape)} does not fit a {H} x {W} alpha: tile sides must be positive")
    grid = (Th, Tw, -(-H // Th), -(-W // Tw))
    if (Th, Tw) != (padded(H), padded(W)) and (max(Th, Tw) ** 2 * 48 >= 2 ** 31 or tile_grid(H, W, max(Th, Tw)) != grid):
        raise ValueError(f"shape {tuple(shape)} does not fit a {H} x {W} alpha: no tile_grid({H}, {W}, tile) has tiles "
                         f"of {Th} x {Tw}")
    chunk_tiles(Th, Tw)                                  # an untiled image may be too large for any forward pass
    return grid


def chunk_tiles(Th: int, Tw: int) -> int:
    """tiles of Th x Tw per forward pass: count * Th * Tw * 48 < MAX_ELEMENTS; MwaB200Error if not even one fits"""
    per = (MAX_ELEMENTS - 1) // (Th * Tw * 48)
    if per < 1:
        raise _abi.MwaB200Error(f"a tile of {Th} x {Tw} is too large: Th * Tw * 48 must stay below 2^31")
    return per


def _check_size(B: int, H: int, W: int) -> None:
    if H < 1 or W < 1:
        raise ValueError(f"image height and width must be >= 1 (got {H} x {W})")
    if B * padded(H) * padded(W) * 48 >= MAX_ELEMENTS:
        raise _abi.MwaB200Error(f"{B} x {H} x {W} is too large: B * Hp * Wp * 48 must stay below 2^31")


def on_device(t: torch.Tensor, device) -> torch.Tensor:
    """t on the CUDA device (the current one if None): one copy for a CPU tensor, non-blocking when it is pinned"""
    if t.is_cuda and device is None:
        return t
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    if device.type != "cuda":
        raise _abi.MwaB200Error(f"RGBA images are converted on a CUDA device (got {device}); there is no CPU fallback")
    return t.to(device, non_blocking=t.is_pinned())


def staged(t: torch.Tensor, device) -> torch.Tensor:
    """on_device, at an address of whole Words (one RGBA pixel, or 4 alpha samples) for the kernels: a view at another
    offset is copied once"""
    t = on_device(t, device)
    return t.clone() if t.data_ptr() % (4 * t.element_size()) else t


def _name(dtype: torch.dtype) -> str:
    return str(dtype).removeprefix("torch.")


def as_batch(t: torch.Tensor, channels: tuple, what: str, dtype: torch.dtype = torch.uint8) -> torch.Tensor:
    """`dtype` (B, H, W, C) or (H, W, C) with C in `channels`, contiguous, as (B, H, W, C)"""
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{what} must be a torch.Tensor (got {type(t).__name__})")
    if t.dtype != dtype:
        raise _abi.MwaB200Error(f"{what} must be {_name(dtype)} (got {t.dtype})")
    if t.dim() not in (3, 4) or t.shape[-1] not in channels:
        raise ValueError(f"{what} must be (B, H, W, C) or (H, W, C) with C in {channels} (got {tuple(t.shape)})")
    if not t.is_contiguous():
        raise ValueError(f"{what} must be contiguous (interleaved channels, rows back to back)")
    return t if t.dim() == 4 else t.unsqueeze(0)


def _ingest(t: torch.Tensor, device, dtype: torch.dtype, what: str):
    t = as_batch(t, (1, 4), what, dtype)
    B, H, W, C = t.shape
    _check_size(B, H, W)
    t = staged(t, device)
    Hp, Wp = padded(H), padded(W)
    alpha = torch.empty(B, 1, Hp, Wp, dtype=torch.float32, device=t.device)
    image = torch.empty(B, 3, Hp, Wp, dtype=torch.float32, device=t.device) if C == 4 else None
    lib = _abi.load()
    with torch.cuda.device(t.device):
        _abi.check(getattr(lib, what + "_ingest")(t.data_ptr(), _abi.ptr(image), alpha.data_ptr(), B, H, W, C,
                                                  _abi.stream_handle()), what + "_ingest")
    _abi.count_launches(1)
    return image, alpha, (H, W)


_DEPTHS = {torch.uint8: "rgba8", torch.uint16: "rgba16"}


def depth(t, what: str) -> str:
    """the entry points' prefix, "rgba8" or "rgba16", for t's sample type"""
    if not isinstance(t, torch.Tensor):
        raise ValueError(f"{what} must be a torch.Tensor (got {type(t).__name__})")
    if t.dtype not in _DEPTHS:
        raise _abi.MwaB200Error(f"{what} must be uint8 or uint16 (got {t.dtype})")
    return _DEPTHS[t.dtype]


def _tile_range(B: int, H: int, W: int, tile_hw, first: int, count: int):
    """(Th, Tw) checked against the C entry points' rules for tiles [first, first + count) of a B x H x W batch"""
    Th, Tw = (int(v) for v in tile_hw)
    if Th < PAD or Tw < PAD or Th % PAD or Tw % PAD:
        raise ValueError(f"tile sides must be positive multiples of {PAD} (got {Th} x {Tw})")
    total = B * -(-H // Th) * -(-W // Tw)
    if first < 0 or count < 0 or first + count > total:
        raise ValueError(f"tiles [{first}, {first + count}) are not within the {total} tiles of {B} x {H} x {W} "
                         f"in tiles of {Th} x {Tw}")
    if count * Th * Tw * 48 >= 2 ** 31:
        raise _abi.MwaB200Error(f"{count} tiles of {Th} x {Tw} are too large: count * Th * Tw * 48 must stay below 2^31")
    return Th, Tw


def ingest_tiles(t: torch.Tensor, tile_hw, first: int, count: int, device=None):
    """(image, alpha): the fp32 planes (count, 3, Th, Tw) and (count, 1, Th, Tw) of tiles [first, first + count) of
    uint8 or uint16 RGBA (B, H, W, 4) or (H, W, 4) (image None for C = 1, an alpha plane alone); tile n = (b * ty + i) * tx
    + j covers rows i * Th.. and columns j * Tw.. of image b, transparent past the image (tile_grid; DESIGN.md 4.8).  A CPU
    input is copied to `device` once: pass the copy back in for the next range."""
    what = depth(t, "rgba")
    t = as_batch(t, (1, 4), what, t.dtype)
    B, H, W, C = t.shape
    Th, Tw = _tile_range(B, H, W, tile_hw, first, count)
    t = staged(t, device)
    alpha = torch.empty(count, 1, Th, Tw, dtype=torch.float32, device=t.device)
    image = torch.empty(count, 3, Th, Tw, dtype=torch.float32, device=t.device) if C == 4 else None
    lib = _abi.load()
    with torch.cuda.device(t.device):
        _abi.check(getattr(lib, what + "_ingest_tiles")(t.data_ptr(), _abi.ptr(image), alpha.data_ptr(), B, H, W, C, Th,
                                                        Tw, first, count, _abi.stream_handle()), what + "_ingest_tiles")
    _abi.count_launches(1)
    return image, alpha


def egress_tiles(x_hat: torch.Tensor, alpha_in: torch.Tensor, out: torch.Tensor, first: int) -> torch.Tensor:
    """write the pixels of `out` (B, H, W, 4), uint8 or uint16 like the (B, H, W) alpha, that the tiles [first, first +
    count) of the decoder's fp32 x_hat (count, 3, Th, Tw) cover: A = alpha, RGB = rint(clamp(x_hat, 0, 1) * full scale)
    where alpha > 0, else 0.  No other byte of `out` is written, so successive ranges fill one output.  Returns out."""
    _abi.require_cuda_f32(x_hat, "x_hat")
    what = depth(alpha_in, "alpha")
    name = "alpha" + what.removeprefix("rgba")
    dtype = alpha_in.dtype
    if alpha_in.dim() != 3 or not alpha_in.is_contiguous():
        raise ValueError(f"{name} must be contiguous {_name(dtype)} (B, H, W) (got {tuple(alpha_in.shape)})")
    B, H, W = alpha_in.shape
    if x_hat.dim() != 4 or x_hat.shape[1] != 3:
        raise ValueError(f"x_hat must be (count, 3, Th, Tw) (got {tuple(x_hat.shape)})")
    count = x_hat.shape[0]
    Th, Tw = _tile_range(B, H, W, x_hat.shape[2:], first, count)
    if (not isinstance(out, torch.Tensor) or out.dtype != dtype or tuple(out.shape) != (B, H, W, 4)
            or not out.is_contiguous() or out.device != x_hat.device):
        raise ValueError(f"out must be contiguous {_name(dtype)} {(B, H, W, 4)} on {x_hat.device} "
                         f"(got {getattr(out, 'dtype', type(out).__name__)} {tuple(getattr(out, 'shape', ()))})")
    alpha_in = on_device(alpha_in, x_hat.device)
    x_hat = x_hat.contiguous()
    if x_hat.data_ptr() % 16:
        x_hat = x_hat.clone()
    lib = _abi.load()
    with torch.cuda.device(x_hat.device):
        _abi.check(getattr(lib, what + "_egress_tiles")(x_hat.data_ptr(), alpha_in.data_ptr(), out.data_ptr(), B, H, W,
                                                        Th, Tw, first, count, _abi.stream_handle()), what + "_egress_tiles")
    _abi.count_launches(1)
    return out


def _egress(x_hat: torch.Tensor, alpha_in: torch.Tensor, dtype: torch.dtype, what: str) -> torch.Tensor:
    _abi.require_cuda_f32(x_hat, "x_hat")
    name = "alpha" + what.removeprefix("rgba")
    if alpha_in.dtype != dtype or alpha_in.dim() != 3 or not alpha_in.is_contiguous():
        raise ValueError(f"{name} must be contiguous {_name(dtype)} (B, H, W) (got {alpha_in.dtype} {tuple(alpha_in.shape)})")
    B, H, W = alpha_in.shape
    _check_size(B, H, W)
    if tuple(x_hat.shape) != (B, 3, padded(H), padded(W)):
        raise ValueError(f"x_hat must be (B, 3, Hp, Wp) = {(B, 3, padded(H), padded(W))} for alpha {tuple(alpha_in.shape)} "
                         f"(got {tuple(x_hat.shape)})")
    alpha_in = on_device(alpha_in, x_hat.device)
    x_hat = x_hat.contiguous()
    if x_hat.data_ptr() % 16:
        x_hat = x_hat.clone()
    out = torch.empty(B, H, W, 4, dtype=dtype, device=x_hat.device)
    lib = _abi.load()
    with torch.cuda.device(x_hat.device):
        _abi.check(getattr(lib, what + "_egress")(x_hat.data_ptr(), alpha_in.data_ptr(), out.data_ptr(), B, H, W,
                                                  _abi.stream_handle()), what + "_egress")
    _abi.count_launches(1)
    return out


def rgba8_ingest(rgba8: torch.Tensor, device=None):
    """(image, alpha, (H, W)): the fp32 planes of uint8 RGBA (C = 4; image None for C = 1, an alpha plane alone), padded to
    multiples of 64.  A CPU input is copied to `device` (default: the current CUDA device) once."""
    return _ingest(rgba8, device, torch.uint8, "rgba8")


def rgba8_egress(x_hat: torch.Tensor, alpha8: torch.Tensor) -> torch.Tensor:
    """uint8 (B, H, W, 4) from the decoder's fp32 (B, 3, Hp, Wp) x_hat (unclamped) and the uint8 (B, H, W) alpha: A = alpha,
    RGB = rint(clamp(x_hat, 0, 1) * 255) where alpha > 0, else 0"""
    return _egress(x_hat, alpha8, torch.uint8, "rgba8")


def rgba16_ingest(rgba16: torch.Tensor, device=None):
    """rgba8_ingest for uint16 samples: alpha = a / 65535, colour / 65535 premultiplied by the binarised alpha.  For 8-bit
    values v, rgba16 = 257 * v gives exactly rgba8_ingest's planes."""
    return _ingest(rgba16, device, torch.uint16, "rgba16")


def rgba16_egress(x_hat: torch.Tensor, alpha16: torch.Tensor) -> torch.Tensor:
    """uint16 (B, H, W, 4) from the decoder's fp32 (B, 3, Hp, Wp) x_hat (unclamped) and the uint16 (B, H, W) alpha:
    A = alpha, RGB = rint(clamp(x_hat, 0, 1) * 65535) where alpha > 0, else 0"""
    return _egress(x_hat, alpha16, torch.uint16, "rgba16")
