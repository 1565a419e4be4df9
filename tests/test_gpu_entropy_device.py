"""The lane-interleaved bitstream format and its device coder (csrc/rans_dev.cu + <package>/entropy.py, DESIGN.md 4.7).
Every lane segment is defined by the host coder (csrc/rans.cu, itself held by tests/test_entropy.py): the device encoder
must write exactly the host coder's bytes for each lane, the device decoder must read streams assembled from host-written
segments, and the codec's device-format round trip must reconstruct exactly what the host format does.  Header parsing,
format detection and build_indexes are also checked on the CPU."""
import importlib
import os
import re
import struct
import warnings

import numpy as np
import pytest
import torch

from oracle import golden_cases as G

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def ent(pkg):
    return importlib.import_module(pkg.codec.__name__.rsplit(".", 1)[0] + ".entropy")


def _gaussian(ent):
    return ent.gaussian_table(ent.get_scale_table())


def _factorized(pkg):
    torch.manual_seed(0)
    eb = pkg.codec.EntropyBottleneck(6)
    eb.update()
    return eb._table


def _message(table, n, seed):
    """symbols around each row's support, every 97th far outside it (multi-digit escapes)"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, table.cdf.shape[0], n).astype(np.int32)
    half = (table.sizes[idx] - 2) / 2.0
    sym = (np.round(rng.normal(0, 1, n) * np.maximum(half / 4, 0.5)) + table.offsets[idx] + half).astype(np.int32)
    sym[::97] += rng.integers(-70000, 70000, sym[::97].size).astype(np.int32)
    return sym, idx


def _host_stream(ent, table, sym, idx, lanes):
    """the lane format restated: header, then the host coder's stream of each lane's elements"""
    segs = [table.encode(sym[l::lanes], idx[l::lanes]) for l in range(lanes)]
    head = struct.pack("<3I", ent.LANES_MAGIC, 0x80000000 | ent.LANES_VERSION, lanes)
    return head + struct.pack(f"<{lanes}I", *[len(s) for s in segs]) + b"".join(segs)


def _to_dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------------------------------------ CPU: format and indexes
def test_header_constants_match_the_c_header(ent):
    text = open(os.path.join(ROOT, "include", "mwa_b200.h")).read()
    assert int(re.search(r"#define MWA_RANS_LANES_MAGIC (0x[0-9A-Fa-f]+)u", text).group(1), 16) == ent.LANES_MAGIC
    assert int(re.search(r"#define MWA_RANS_LANES_VERSION (\d+)u", text).group(1)) == ent.LANES_VERSION


def test_default_lane_count(ent):
    assert ent.default_lanes(0) == 1 and ent.default_lanes(1) == 1 and ent.default_lanes(16384) == 1
    assert ent.default_lanes(16385) == 2
    assert ent.default_lanes(80 * 64 * 96) == 30 and ent.default_lanes(192 * 8 * 12) == 2     # y and z at 768 x 512
    assert ent.default_lanes(10 ** 9) == 1024


def test_malformed_headers_raise_before_any_launch(ent):
    table = _gaussian(ent)
    sym, idx = _message(table, 300, 3)
    good = _host_stream(ent, table, sym, idx, 3)
    assert ent.is_device_stream(good)
    assert list(ent.parse_lanes(good)) == [len(table.encode(sym[l::3], idx[l::3])) for l in range(3)]
    words = list(struct.unpack(f"<{len(good) // 4}I", good))

    def patched(**kw):
        w = list(words)
        for k, v in kw.items():
            w[int(k[1:])] = v
        return struct.pack(f"<{len(w)}I", *w)

    bad = {
        "bad magic": patched(w0=words[0] ^ 1),
        "bad version": patched(w1=0x80000002),
        "zero lanes": patched(w2=0),
        "lane count beyond the string": patched(w2=10 ** 6),
        "length not a multiple of 4": patched(w3=words[3] + 2, w4=words[4] - 2),
        "length below 8": patched(w3=4, w4=words[4] + words[3] - 4),
        "lengths do not add up": patched(w3=words[3] + 4),
        "truncated string": good[:-4],
        "ragged string": good + b"\0",
        "header only": good[:10],
    }
    for s in bad.values():
        with pytest.raises(ValueError):
            ent.parse_lanes(s)
        # the device decoder's constructor parses before it touches the device
        with pytest.raises(ValueError):
            ent.LaneStreams([[good, s]], "cuda")


def test_host_streams_are_never_taken_for_device_streams(pkg, ent):
    tables = [_gaussian(ent), _factorized(pkg)]
    rng = np.random.default_rng(5)
    for k in range(400):
        table = tables[k % 2]
        sym, idx = _message(table, int(rng.integers(0, 3000)), k)
        s = table.encode(sym, idx)
        assert len(s) >= 8 and not ent.is_device_stream(s)
        assert ent.stream_format([s]) == "host"
    empty = tables[0].encode(np.zeros(0, np.int32), np.zeros(0, np.int32))
    assert len(empty) == 8 and not ent.is_device_stream(empty)
    dev = _host_stream(ent, tables[0], *_message(tables[0], 10, 0), 2)
    with pytest.raises(ValueError, match="mixed"):
        ent.stream_format([empty, dev])


def _old_build_indexes(scales, scale_table):
    """build_indexes as it was: 63 minus the number of table scales (all but the last) >= the bounded scale"""
    table = scale_table.to(scales.device)
    s = torch.clamp_min(scales, 0.11)
    idx = torch.full(s.shape, len(table) - 1, dtype=torch.int32, device=scales.device)
    for v in table[:-1].tolist():
        idx -= (s <= v).to(torch.int32)
    return idx


def _check_build_indexes(ent, device):
    st = ent.get_scale_table()
    g = torch.Generator().manual_seed(9)
    special = torch.tensor([0.0, -1.0, 0.05, 0.11, 0.1100001, 255.9, 256.0, 257.0, 1e30, float("inf"), float("-inf"),
                            float("nan")])
    scales = torch.cat([torch.exp(torch.rand(20000, generator=g) * 7 - 3), st, special]).view(4, -1)
    scales = scales.to(device)
    new = ent.build_indexes(scales, st)
    assert new.dtype == torch.int32 and new.device == scales.device
    assert torch.equal(new, _old_build_indexes(scales, st))
    assert int(new.view(-1)[-1]) == 63 and int(new.view(-1)[-4]) == 63 and int(new.view(-1)[-3]) == 63   # nan, +inf, 1e30


def test_build_indexes_equals_the_loop_on_the_cpu(ent):
    _check_build_indexes(ent, "cpu")


@gpu
def test_build_indexes_equals_the_loop_on_cuda(ent, cuda_dev):
    _check_build_indexes(ent, cuda_dev)


# ------------------------------------------------------------------------------------------------ GPU: coder
@gpu
@pytest.mark.parametrize("which", ["gaussian", "factorized"])
@pytest.mark.parametrize("n", [0, 1, 1000, 50000])
@pytest.mark.parametrize("lanes", [1, 5, 32, 300])
def test_lanes_equal_the_host_coder(pkg, ent, cuda_dev, which, n, lanes):
    table = _gaussian(ent) if which == "gaussian" else _factorized(pkg)
    msgs = [_message(table, n, seed) for seed in (1, 2)]
    sym = np.stack([m[0] for m in msgs])
    idx = np.stack([m[1] for m in msgs])
    got = table.encode_lanes(_to_dev(sym), _to_dev(idx), lanes).strings()
    assert len(got) == 2
    for s in range(2):
        assert ent.is_device_stream(got[s])
        assert got[s] == _host_stream(ent, table, sym[s], idx[s], lanes)


@gpu
def test_encoder_retries_when_escapes_overflow_the_slots(ent, cuda_dev):
    table = _gaussian(ent)
    rng = np.random.default_rng(4)
    n = 4000
    idx = np.zeros(n, np.int32)                              # the narrowest table: everything else escapes
    sym = rng.integers(-2 ** 26, 2 ** 26, n).astype(np.int32)
    enc = table.encode_lanes(_to_dev(sym[None]), _to_dev(idx[None]), 3)
    first = enc.slot_words
    got = enc.strings()
    assert enc.slot_words > first
    assert got[0] == _host_stream(ent, table, sym, idx, 3)


@gpu
def test_invalid_index_raises(ent, cuda_dev):
    table = _gaussian(ent)
    sym, idx = _message(table, 100, 1)
    idx[50] = 64
    with pytest.raises(ent._abi.MwaB200Error, match="invalid"):
        table.encode_lanes(_to_dev(sym[None]), _to_dev(idx[None]), 4).strings()


@gpu
@pytest.mark.parametrize("lanes", [None, 32])
def test_decode_in_uneven_pieces(ent, cuda_dev, lanes):
    table = _gaussian(ent)
    n = 50000
    msgs = [_message(table, n, seed) for seed in (6, 7, 8)]
    sym = np.stack([m[0] for m in msgs])
    idx = np.stack([m[1] for m in msgs])
    strings = table.encode_lanes(_to_dev(sym), _to_dev(idx), lanes).strings()
    streams = ent.LaneStreams([strings], cuda_dev)
    dec = streams.decoder(table, 0)
    cuts = [0, 1, 12345, n]
    out = [dec.decode(_to_dev(idx[:, a:b])) for a, b in zip(cuts[:-1], cuts[1:])]
    streams.check()
    assert np.array_equal(torch.cat(out, 1).cpu().numpy(), sym)


@gpu
def test_decode_streams_with_different_lane_counts_and_host_written_segments(pkg, ent, cuda_dev):
    """one call over streams of 1, 7, 300 and 64 lanes; the last two assembled on the host from host-coder segments only
    (this pins the decoder independently of the device encoder).  A second group with another table rides in the same
    staging copy."""
    table, fact = _gaussian(ent), _factorized(pkg)
    n = 20000
    msgs = [_message(table, n, seed) for seed in (10, 11, 12, 13)]
    strings = [table.encode_lanes(_to_dev(m[0][None]), _to_dev(m[1][None]), L).strings()[0]
               for m, L in zip(msgs[:2], (1, 7))]
    strings += [_host_stream(ent, table, m[0], m[1], L) for m, L in zip(msgs[2:], (300, 64))]
    fsym, fidx = _message(fact, 999, 14)
    streams = ent.LaneStreams([strings, [_host_stream(ent, fact, fsym, fidx, 5)]], cuda_dev)
    dec, fdec = streams.decoder(table, 0), streams.decoder(fact, 1)
    idx = np.stack([m[1] for m in msgs])
    half = n // 2
    out = torch.cat([dec.decode(_to_dev(idx[:, :half])), dec.decode(_to_dev(idx[:, half:]))], 1)
    fout = fdec.decode(_to_dev(fidx[None]))
    streams.check()
    assert np.array_equal(out.cpu().numpy(), np.stack([m[0] for m in msgs]))
    assert np.array_equal(fout.cpu().numpy()[0], fsym)


@gpu
def test_truncated_segment_sets_the_status(ent, cuda_dev):
    table = _gaussian(ent)
    sym, idx = _message(table, 5000, 15)
    good = _host_stream(ent, table, sym, idx, 4)
    lengths = ent.parse_lanes(good)
    words = list(struct.unpack(f"<{len(good) // 4}I", good))
    # drop the last word of lane 2's segment and shorten its length to match: the header stays well formed
    end = 3 + 4 + int(lengths[:3].sum()) // 4
    words[3 + 2] -= 4
    del words[end - 1]
    bad = struct.pack(f"<{len(words)}I", *words)
    ent.parse_lanes(bad)
    streams = ent.LaneStreams([[good, bad]], cuda_dev)
    dec = streams.decoder(table, 0)
    out = dec.decode(_to_dev(np.stack([idx, idx])))
    with pytest.raises(ent._abi.MwaB200Error, match=r"\[1\]"):
        streams.check()
    assert np.array_equal(out[0].cpu().numpy(), sym)


@gpu
def test_coder_captures_in_a_cuda_graph(ent, cuda_dev):
    """no host synchronisation inside encode or decode: both capture, and replays reproduce the eager results"""
    table = _gaussian(ent)
    n = 30000
    msgs = [_message(table, n, seed) for seed in (16, 17)]
    sym = _to_dev(np.stack([m[0] for m in msgs]))
    idx = _to_dev(np.stack([m[1] for m in msgs]))
    eager = table.encode_lanes(sym, idx, 24).strings()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        table.encode_lanes(sym, idx, 24)                         # warm-up on the capture stream's side
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enc = table.encode_lanes(sym, idx, 24)
    slot_words = enc.slot_words
    for _ in range(2):
        enc.out.zero_()
        g.replay()
        assert enc.strings() == eager and enc.slot_words == slot_words

    streams = ent.LaneStreams([eager], cuda_dev)
    state0 = streams.state.clone()
    pieces = [idx[:, :7].contiguous(), idx[:, 7:20000].contiguous(), idx[:, 20000:].contiguous()]
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        streams.state.copy_(state0)
        streams.status.zero_()
        dec = streams.decoder(table, 0)
        outs = [dec.decode(p) for p in pieces]
    for _ in range(2):
        for o in outs:
            o.fill_(-1)
        g2.replay()
        streams.check()
        assert torch.equal(torch.cat(outs, 1), sym)


@gpu
def test_entropy_bottleneck_device_round_trip(pkg, ent, cuda_dev):
    torch.manual_seed(0)
    eb = pkg.codec.EntropyBottleneck(6)
    with torch.no_grad():
        eb.quantiles[:, 0, 1] = torch.linspace(-0.3, 0.4, 6)
        eb.quantiles[:, 0, 0] = -4.0
        eb.quantiles[:, 0, 2] = 5.0
    eb = eb.to(cuda_dev)
    z = (torch.randn(3, 6, 5, 7) * 6).to(cuda_dev)
    strings = eb.compress(z, coder="device", lanes=4)
    assert len(strings) == 3 and all(ent.is_device_stream(s) for s in strings)
    want = torch.round(z - eb._get_medians()) + eb._get_medians()
    assert torch.equal(eb.decompress(strings, (5, 7)), want)
    host = eb.compress(z)
    assert torch.equal(eb.decompress(host, (5, 7)), want)
    with pytest.raises(ValueError, match="mixed"):
        eb.decompress([host[0], strings[1], host[2]], (5, 7))
    with pytest.raises(ValueError):
        eb.compress(z, coder="gpu")
    with pytest.raises(ent._abi.MwaB200Error, match="CUDA"):
        pkg.codec.EntropyBottleneck(6).compress(z.cpu(), coder="device")


# ------------------------------------------------------------------------------------------------ GPU: the codec
def _codec(pkg, model_keys, seed, dev):
    net = pkg.RGBACodec().eval()
    net.load_state_dict(G.model_state(model_keys, seed), strict=False)
    return net.to(dev)


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
def test_codec_device_format_round_trip(pkg, ent, cuda_dev, model_keys):
    """the case of test_compress_decompress_round_trip: the device format reconstructs exactly what the host format and
    the forward do, at a size overhead of at most 16 bytes a lane + 16 a string"""
    cfg = next(iter(G.MODEL_CASES.values()))
    p = G.model_inputs(cfg)
    net = _codec(pkg, model_keys, cfg["seed"], cuda_dev)
    image = torch.cat([p["image"], p["image"].flip(3)], 0).to(cuda_dev)
    alpha = torch.cat([p["alpha"], p["alpha"].flip(3)], 0).to(cuda_dev)
    with torch.no_grad():
        host = net.compress(image, alpha)
        rec_host = net.decompress(host["strings"], host["shape"], alpha)["x_hat"]
        me = net.EncMakeMask(alpha)
        x_hat = net(image, alpha, alpha, me[0], me[1], me[2], me[3])[0]
    assert torch.equal(rec_host, x_hat.clamp(0, 1))
    for lanes in (None, 7, 64):
        with torch.no_grad():
            out = net.compress(image, alpha, coder="device", lanes=lanes)
            assert tuple(out["shape"]) == tuple(host["shape"])
            rec = net.decompress(out["strings"], out["shape"], alpha)["x_hat"]
        assert torch.equal(rec, rec_host) and torch.equal(rec, x_hat.clamp(0, 1))
        hz, wz = out["shape"]
        for group, host_group, n in zip(out["strings"], host["strings"], (net.M * 64 * hz * wz, 192 * hz * wz)):
            assert len(group) == 2
            for s, h in zip(group, host_group):
                L = len(ent.parse_lanes(s))
                assert L == (lanes or ent.default_lanes(n))
                assert len(s) <= len(h) + 16 * L + 16, (len(s), len(h), L)
    with torch.no_grad(), pytest.raises(ValueError, match="mixed"):
        net.decompress([host["strings"][0], out["strings"][1]], host["shape"], alpha)


@gpu
def test_device_decompress_synchronises_once(pkg, cuda_dev, model_keys):
    cfg = next(iter(G.MODEL_CASES.values()))
    p = G.model_inputs(cfg)
    net = _codec(pkg, model_keys, cfg["seed"], cuda_dev)
    image, alpha = p["image"].to(cuda_dev), p["alpha"].to(cuda_dev)
    with torch.no_grad():
        dev_out = net.compress(image, alpha, coder="device")
        host_out = net.compress(image, alpha)
        for out in (dev_out, host_out):                          # warm-up: tables on the device, kernels loaded
            net.decompress(out["strings"], out["shape"], alpha)
        torch.cuda.synchronize()
        on_dev = _syncs(lambda: net.decompress(dev_out["strings"], dev_out["shape"], alpha))
        on_host = _syncs(lambda: net.decompress(host_out["strings"], host_out["shape"], alpha))
    assert len(on_dev) <= 1, on_dev
    assert len(on_host) >= net.num_slices, on_host
