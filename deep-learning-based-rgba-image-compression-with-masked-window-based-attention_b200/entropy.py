"""Entropy-coding side of the codec (SURVEY.md section 8f, rank 4): quantised CDF tables of the two entropy models, the
binding of the host rANS coder (csrc/rans.cu) and of the lane-interleaved device coder (csrc/rans_dev.cu, DESIGN.md 4.7).

Reference call sites: models/AutoEncoderRGB_Journal.py:306-311 (update), :319-320 (entropy_bottleneck.compress /
decompress), :330-368 / :374-403 (BufferedRansEncoder / RansDecoder with the Gaussian conditional's tables).  The classes
behind them are CompressAI's (third-party, absent, unversioned): the table construction below restates their published
definitions (scale table exp(linspace(log 0.11, log 256, 64)), tail mass 1e-9, 16-bit CDFs with every symbol given a
non-zero frequency) -- enough for a self-consistent bitstream; byte parity with CompressAI is UNPINNED.
"""
from __future__ import annotations

import ctypes
import math
import struct

import numpy as np
import torch

from . import _abi

PRECISION = 16
SCALES_MIN, SCALES_MAX, SCALES_LEVELS = 0.11, 256.0, 64
TAIL_MASS = 1e-9
# -norm.ppf(TAIL_MASS / 2): how many standard deviations the tabulated support reaches
TAIL_MULTIPLIER = 6.109410204869


def get_scale_table(lo=SCALES_MIN, hi=SCALES_MAX, levels=SCALES_LEVELS) -> torch.Tensor:
    """models/AutoEncoderRGB_Journal.py:23-27"""
    return torch.exp(torch.linspace(math.log(lo), math.log(hi), levels))


def pmf_to_quantized_cdf(pmf: np.ndarray, precision: int = PRECISION) -> np.ndarray:
    """frequencies proportional to pmf summing to 2^precision, none of them zero (a zero is filled by taking one count from
    the smallest frequency above 1, as CompressAI's pmf_to_quantized_cdf does)"""
    freq = np.round(np.asarray(pmf, dtype=np.float64) * (1 << precision)).astype(np.int64)
    total = int(freq.sum())
    if total <= 0:
        raise ValueError("pmf_to_quantized_cdf: empty distribution")
    cdf = np.concatenate([[0], np.cumsum(freq)])
    cdf = ((1 << precision) * cdf) // total
    cdf[-1] = 1 << precision
    n = len(cdf) - 1
    for i in range(n):
        if cdf[i] == cdf[i + 1]:
            f = np.diff(cdf)
            cand = np.where(f > 1)[0]
            if cand.size == 0:
                raise ValueError("pmf_to_quantized_cdf: more symbols than counts")
            j = int(cand[np.argmin(f[cand])])
            if j < i:
                cdf[j + 1:i + 1] -= 1
            else:
                cdf[i + 1:j + 1] += 1
    assert np.all(np.diff(cdf) > 0) and cdf[0] == 0 and cdf[-1] == 1 << precision
    return cdf.astype(np.int32)


class CdfTable:
    """(ncdf, max_len) int32 quantised CDFs + per-row length and symbol offset, on the host (the coder runs there)"""

    def __init__(self, pmfs, tail_masses, lengths, offsets):
        n, max_len = len(lengths), int(max(lengths)) + 2
        self.cdf = np.zeros((n, max_len), dtype=np.int32)
        for i in range(n):
            prob = np.concatenate([np.asarray(pmfs[i][:lengths[i]], dtype=np.float64), [float(tail_masses[i])]])
            c = pmf_to_quantized_cdf(prob)
            self.cdf[i, :len(c)] = c
        self.sizes = (np.asarray(lengths, dtype=np.int32) + 2).astype(np.int32)
        self.offsets = np.asarray(offsets, dtype=np.int32)
        self._device_copies = {}

    def _p(self, a):
        return a.ctypes.data_as(ctypes.c_void_p)

    def encode(self, symbols: np.ndarray, indexes: np.ndarray) -> bytes:
        lib = _abi.load()
        symbols = np.ascontiguousarray(symbols, dtype=np.int32).reshape(-1)
        indexes = np.ascontiguousarray(indexes, dtype=np.int32).reshape(-1)
        cap = 16 + 8 * symbols.size + 64
        while True:
            out = np.empty(cap, dtype=np.uint8)
            n = lib.rans_encode_with_indexes(self._p(symbols), self._p(indexes), symbols.size, self._p(self.cdf),
                                             self.cdf.shape[1], self._p(self.sizes), self._p(self.offsets), self.cdf.shape[0],
                                             self._p(out), cap)
            if n == -4:                       # MWA_ERR_WORKSPACE: heavy use of the escape code; retry with more room
                cap *= 4
                continue
            if n < 0:
                _abi.check(int(n), "rans_encode_with_indexes")
            return out[:n].tobytes()

    def decoder(self, stream: bytes) -> "StreamDecoder":
        return StreamDecoder(self, stream)

    def on_device(self, device: torch.device):
        """(cdf, sizes, offsets) as int32 tensors on `device`, uploaded once"""
        device = torch.device(device)
        if device.type != "cuda":
            raise _abi.MwaB200Error(f"the device coder needs a CUDA device (got {device}); this package is sm_100a-only "
                                    "and has no CPU fallback")
        key = device.index if device.index is not None else torch.cuda.current_device()
        if key not in self._device_copies:
            self._device_copies[key] = tuple(torch.from_numpy(a).to(device) for a in (self.cdf, self.sizes, self.offsets))
        return self._device_copies[key]

    def encode_lanes(self, symbols: torch.Tensor, indexes: torch.Tensor, lanes: int | None = None) -> "LaneEncoding":
        """Lane-format streams, one per row of the (S, n) int32 CUDA tensors `symbols` / `indexes`, coded on the GPU with
        `lanes` lanes per stream (default_lanes(n) if None).  Launches only; .strings() of the result waits for them."""
        return LaneEncoding(self, symbols, indexes, default_lanes(symbols.shape[-1]) if lanes is None else int(lanes))


class StreamDecoder:
    """RansDecoder.set_stream + decode_stream: successive calls continue on the same stream"""

    def __init__(self, table: CdfTable, stream: bytes):
        self.t, self.buf = table, np.frombuffer(stream, dtype=np.uint8).copy()
        self.state = np.zeros(4, dtype=np.int64)

    def decode(self, indexes: np.ndarray) -> np.ndarray:
        lib = _abi.load()
        t = self.t
        indexes = np.ascontiguousarray(indexes, dtype=np.int32).reshape(-1)
        out = np.empty(indexes.size, dtype=np.int32)
        _abi.check(lib.rans_decode_with_indexes(t._p(self.buf), self.buf.size, t._p(self.state), t._p(indexes), indexes.size,
                                                t._p(t.cdf), t.cdf.shape[1], t._p(t.sizes), t._p(t.offsets), t.cdf.shape[0],
                                                t._p(out)), "rans_decode_with_indexes")
        return out


# ------------------------------------------------------------------------------------------------ lane-interleaved format
# One stream per image, little-endian u32 words: LANES_MAGIC, 0x80000000 | LANES_VERSION, L, the byte lengths of the L lane
# segments, the segments.  Element g of the message belongs to lane g mod L; a segment is exactly what the host coder
# writes for its lane's elements.  Constants: include/mwa_b200.h (MWA_RANS_LANES_MAGIC, MWA_RANS_LANES_VERSION).
LANES_MAGIC = 0x4C41574D                  # "MWAL"
LANES_VERSION = 1
SYMBOLS_PER_LANE = 16384                  # default lane count: one lane per this many symbols ...
MAX_DEFAULT_LANES = 1024                  # ... up to this many
_HEADER_WORDS = 3


def default_lanes(n: int) -> int:
    """clamp(ceil(n / 16384), 1, 1024): 30 lanes for a 768 x 512 image's y, 2 for its z"""
    return min(max(-(-int(n) // SYMBOLS_PER_LANE), 1), MAX_DEFAULT_LANES)


def is_device_stream(stream: bytes) -> bool:
    """True for the lane-interleaved format.  Its word 1 is 0x80000000 | version.  In a host-format stream word 1 is the
    high half of the encoder's final 64-bit state, which stays in [2^31, 2^63), so it is always < 2^31, and a host stream
    is always at least 8 bytes long: the top bit of byte 7 tells the two formats apart with no ambiguity."""
    return len(stream) >= 8 and (stream[7] & 0x80) != 0


def stream_format(strings) -> str:
    """'device' or 'host' for a set of strings decoded together; mixed formats raise"""
    kinds = {is_device_stream(s) for s in strings}
    if len(kinds) > 1:
        raise ValueError("host-format and device-format (lane-interleaved) strings mixed in one call")
    return "device" if kinds == {True} else "host"


def parse_lanes(stream: bytes) -> np.ndarray:
    """byte lengths (int64) of the lane segments of a lane-format stream; ValueError on a malformed header"""
    if len(stream) < 4 * _HEADER_WORDS or len(stream) % 4:
        raise ValueError(f"lane-format stream of {len(stream)} bytes: too short or not whole words")
    magic, version, lanes = struct.unpack_from("<3I", stream)
    if magic != LANES_MAGIC:
        raise ValueError(f"lane-format stream: bad magic {magic:#010x}")
    if version != 0x80000000 | LANES_VERSION:
        raise ValueError(f"lane-format stream: unsupported version word {version:#010x}")
    if lanes == 0:
        raise ValueError("lane-format stream: zero lanes")
    if 4 * (_HEADER_WORDS + lanes) > len(stream):
        raise ValueError(f"lane-format stream: {lanes} lane lengths do not fit in {len(stream)} bytes")
    lengths = np.frombuffer(stream, dtype="<u4", count=lanes, offset=4 * _HEADER_WORDS).astype(np.int64)
    if np.any(lengths % 4) or np.any(lengths < 8):
        raise ValueError("lane-format stream: a lane length is not a multiple of 4 or below 8")
    if 4 * (_HEADER_WORDS + lanes) + int(lengths.sum()) != len(stream):
        raise ValueError("lane-format stream: lane lengths do not add up to the stream's size")
    return lengths


def _require_int32_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise _abi.MwaB200Error(f"{name} must be a CUDA tensor (got {t.device}); this package is sm_100a-only "
                                "and has no CPU fallback")
    if t.dtype != torch.int32 or t.dim() != 2 or not t.is_contiguous():
        raise _abi.MwaB200Error(f"{name} must be a contiguous (streams, n) int32 tensor (got {t.dtype}, {tuple(t.shape)})")


class LaneEncoding:
    """rans_lanes_encode + rans_lanes_pack launched on the current stream; strings() waits for them"""

    def __init__(self, table: CdfTable, symbols: torch.Tensor, indexes: torch.Tensor, lanes: int, slot_words: int = 0):
        _require_int32_cuda(symbols, "symbols")
        _require_int32_cuda(indexes, "indexes")
        if symbols.shape != indexes.shape or symbols.device != indexes.device:
            raise ValueError("symbols and indexes must have the same shape and device")
        if lanes < 1:
            raise ValueError(f"lanes must be >= 1 (got {lanes})")
        self.t, self.symbols, self.indexes, self.lanes = table, symbols, indexes, lanes
        # without escapes a symbol costs at most 16 bits: half a word per element a lane holds; retried larger otherwise
        self.slot_words = slot_words or -(-symbols.shape[1] // lanes) // 2 + 16
        self._launch()

    def _launch(self):
        lib = _abi.load()
        S, n = self.symbols.shape
        L, sw, dev = self.lanes, self.slot_words, self.symbols.device
        cdf, sizes, offsets = self.t.on_device(dev)
        slots = torch.empty(S * L * sw, dtype=torch.int32, device=dev)
        lane_words = torch.empty(S * L, dtype=torch.int32, device=dev)
        lane_dst = torch.empty(S * L, dtype=torch.int64, device=dev)
        self.out = torch.empty(max(S * (_HEADER_WORDS + L + L * sw), 1), dtype=torch.int32, device=dev)
        self.stream_bytes = torch.empty(S + 1, dtype=torch.int64, device=dev)
        if S == 0:
            self.stream_bytes.zero_()
            return
        with torch.cuda.device(dev):
            h = _abi.stream_handle()
            _abi.check(lib.rans_lanes_encode(self.symbols.data_ptr(), self.indexes.data_ptr(), S, n, L, cdf.data_ptr(),
                                             cdf.shape[1], sizes.data_ptr(), offsets.data_ptr(), cdf.shape[0],
                                             slots.data_ptr(), sw, lane_words.data_ptr(), h), "rans_lanes_encode")
            _abi.check(lib.rans_lanes_pack(slots.data_ptr(), sw, lane_words.data_ptr(), S, L, lane_dst.data_ptr(),
                                           self.stream_bytes.data_ptr(), self.out.data_ptr(), self.out.numel(), h),
                       "rans_lanes_pack")
        _abi.count_launches(3)

    def strings(self) -> list[bytes]:
        """the streams as bytes: one small copy of their lengths, then one copy of all of them"""
        while True:
            info = self.stream_bytes.cpu().numpy()
            total = int(info[-1])
            if total != -4:                   # MWA_ERR_WORKSPACE: heavy use of the escape code; retry with more room
                break
            self.slot_words *= 4
            self._launch()
        if total < 0:
            _abi.check(total, "rans_lanes_encode")
        host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
        host.copy_(self.out.view(torch.uint8)[:total], non_blocking=True)
        torch.cuda.current_stream(self.out.device).synchronize()
        data = host.numpy().tobytes()
        ends = np.cumsum(info[:-1])
        return [data[end - size:end] for size, end in zip(info[:-1].tolist(), ends.tolist())]


class LaneStreams:
    """Lane-format strings, in groups decoded with different tables, parsed and checked on the host, then staged on the
    device in one pinned, non-blocking copy: lane states, lanes per stream and the stream words.  Every stream has a
    status word on the device; check() reads them all in one synchronisation."""

    def __init__(self, groups, device):
        device = torch.device(device)
        if device.type != "cuda":
            raise _abi.MwaB200Error(f"the device decoder needs a CUDA device (got {device}); this package is sm_100a-only "
                                    "and has no CPU fallback")
        groups = [list(g) for g in groups]
        parsed = [[parse_lanes(s) for s in g] for g in groups]
        n_streams = sum(len(g) for g in groups)
        n_lanes = sum(len(p) for g in parsed for p in g)
        data_words = sum(len(s) for g in groups for s in g) // 4
        state = np.zeros((n_lanes, 4), dtype=np.int64)
        stream_lanes = np.zeros(n_streams + (n_streams & 1), dtype=np.int32)      # padded to 8 bytes
        self.groups = []                       # (first lane row, lanes, first stream, streams) per group
        row = stream = word = 0
        for g, p in zip(groups, parsed):
            self.groups.append((row, sum(len(x) for x in p), stream, len(g)))
            for local, (s, lengths) in enumerate(zip(g, p)):
                seg = word + _HEADER_WORDS + len(lengths) + np.concatenate([[0], np.cumsum(lengths // 4)])
                rows = slice(row, row + len(lengths))
                state[rows, 1], state[rows, 2] = seg[:-1], seg[1:]
                state[rows, 3] = local + (np.arange(len(lengths), dtype=np.int64) << 32)
                stream_lanes[stream] = len(lengths)
                row, stream, word = row + len(lengths), stream + 1, word + len(s) // 4
        head = state.tobytes() + stream_lanes.tobytes()
        host = torch.empty(len(head) + 4 * data_words, dtype=torch.uint8, pin_memory=True)
        hv = host.numpy()
        hv[:len(head)] = np.frombuffer(head, dtype=np.uint8)
        hv[len(head):] = np.frombuffer(b"".join(s for g in groups for s in g), dtype=np.uint8)
        staged = host.to(device, non_blocking=True)
        self._host = host                      # the copy reads it asynchronously
        a, b = state.nbytes, state.nbytes + stream_lanes.nbytes
        self.state = staged[:a].view(torch.int64).view(n_lanes, 4)
        self.stream_lanes = staged[a:b].view(torch.int32)
        self.data = staged[b:].view(torch.int32)
        self.status = torch.zeros(n_streams, dtype=torch.int32, device=device)
        self.device = device

    def decoder(self, table: CdfTable, group: int) -> "LaneDecoder":
        return LaneDecoder(self, table, group)

    def check(self) -> None:
        """raises MwaB200Error if any stream was truncated or corrupt (the one synchronisation of a device decode)"""
        bad = np.flatnonzero(self.status.cpu().numpy())
        if bad.size:
            raise _abi.MwaB200Error(f"rans_lanes_decode: truncated or corrupt lane-format stream(s) {bad.tolist()}")


class LaneDecoder:
    """RansDecoder.set_stream + decode_stream for one group of a LaneStreams, all its streams at once: successive decode()
    calls continue where the last one stopped.  Launches only; LaneStreams.check() reports failures."""

    def __init__(self, streams: LaneStreams, table: CdfTable, group: int):
        self.s, self.t = streams, table
        self.row, self.lanes, self.first, self.count = streams.groups[group]
        self.position = 0

    def decode(self, indexes: torch.Tensor) -> torch.Tensor:
        """(streams, n) int32 CUDA indexes of the next n elements of every stream -> their (streams, n) int32 symbols"""
        _require_int32_cuda(indexes, "indexes")
        if indexes.shape[0] != self.count:
            raise ValueError(f"indexes has {indexes.shape[0]} rows for {self.count} streams")
        lib = _abi.load()
        s, dev = self.s, self.s.device
        cdf, sizes, offsets = self.t.on_device(dev)
        n = indexes.shape[1]
        out = torch.empty(self.count, n, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _abi.check(lib.rans_lanes_decode(s.data.data_ptr(), s.data.numel(), s.state[self.row:].data_ptr(), self.lanes,
                                             s.stream_lanes[self.first:].data_ptr(), self.count, indexes.data_ptr(), n,
                                             self.position, cdf.data_ptr(), cdf.shape[1], sizes.data_ptr(),
                                             offsets.data_ptr(), cdf.shape[0], out.data_ptr(),
                                             s.status[self.first:].data_ptr(), _abi.stream_handle()), "rans_lanes_decode")
        _abi.count_launches(1)
        self.position += n
        return out


def _std_cumulative(x: torch.Tensor) -> torch.Tensor:
    return 0.5 * torch.erfc(-(2 ** -0.5) * x)


def gaussian_table(scale_table: torch.Tensor) -> CdfTable:
    """GaussianConditional.update_scale_table / update: one CDF per scale level, support +- ceil(6.1 scale)"""
    st = scale_table.double().cpu()
    center = torch.ceil(st * TAIL_MULTIPLIER).long()
    length = 2 * center + 1
    max_len = int(length.max())
    samples = torch.abs(torch.arange(max_len).double()[None, :] - center[:, None].double())
    s = st[:, None]
    upper, lower = _std_cumulative((0.5 - samples) / s), _std_cumulative((-0.5 - samples) / s)
    pmf = (upper - lower).numpy()
    tail = (2 * lower[:, 0]).numpy()
    return CdfTable(pmf, tail, length.tolist(), (-center).tolist())


def build_indexes(scales: torch.Tensor, scale_table: torch.Tensor) -> torch.Tensor:
    """GaussianConditional.build_indexes: index of the first table scale >= max(scale, lower bound), i.e. the number of
    table scales below it; the last index for anything above the table, +inf and NaN included.  One launch, no host
    synchronisation."""
    table = scale_table.to(device=scales.device, dtype=scales.dtype)
    return torch.bucketize(torch.clamp_min(scales, SCALES_MIN), table[:-1], out_int32=True)
