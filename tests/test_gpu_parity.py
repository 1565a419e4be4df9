"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Every check goes through the product's public
API (nn.Module -> ctypes -> C ABI -> sm_100a kernels) and compares with the CPU oracle / the committed
outputs of the reference.  Tolerance for floating-point results: BASELINE.json's 1e-3 relative / 1e-4 absolute;
the SIMT kernels (plain fp32) are held to a much tighter bound.  Rounded latents are bit-exact.
"""
import numpy as np
import pytest
import torch

from oracle import golden_cases as G
from oracle import ref_ops as R

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-3, 1e-4          # north_star tolerance
ALGOS = {"auto": 0, "simt": 1}


def _t(a):
    return torch.from_numpy(np.asarray(a))


def _mk_attn(pkg, cfg, p, dev, masked=None):
    masked = cfg["masked"] if masked is None else masked
    cls = pkg.MaskedWinBasedAttention if masked else pkg.WinBasedAttention
    m = cls(dim=cfg["C"], num_heads=cfg["heads"], window_size=cfg["ws"], shift_size=cfg["shift"],
            qkv_bias=cfg.get("qkv_bias", True))
    with torch.no_grad():
        m.attn.qkv.weight.copy_(p["qkv_w"])
        if p["qkv_b"] is not None:
            m.attn.qkv.bias.copy_(p["qkv_b"])
        m.attn.proj.weight.copy_(p["proj_w"])
        m.attn.proj.bias.copy_(p["proj_b"])
        m.attn.relative_position_bias_table.copy_(p["table"])
    return m.to(dev)


def _oracle_attn(cfg, p, dtype=torch.float32):
    c = lambda t: None if t is None else t.to(dtype)
    return R.masked_window_attention(c(p["x"]), c(p["alpha"]), c(p["qkv_w"]), c(p["qkv_b"]), c(p["proj_w"]),
                                     c(p["proj_b"]), c(p["table"]), cfg["heads"], cfg["ws"], cfg["shift"])


def _check_attention(y, p, cfg, algo, ref32=None):
    """Every kernel selection the modules make by default is fp32-faithful: the auto path (split-precision tcgen05 kernel
    for 8x8 / C=192, fp32 small-window kernel for 4x4 / C=80, general SIMT kernel otherwise) is held to BASELINE.json's
    1e-3 relative / 1e-4 absolute against the fp64 oracle AND against the committed outputs of the reference itself, on
    every element -- also on these deliberately harsh weights (logit std ~5).  The forced SIMT kernel is held tighter."""
    ref64 = _oracle_attn(cfg, p, torch.float64)
    y = y.double().cpu()
    rt, at = (RTOL, ATOL) if algo == "auto" else (1e-4, 2e-5)
    torch.testing.assert_close(y, ref64, rtol=rt, atol=at)
    if ref32 is not None:
        torch.testing.assert_close(y.float(), ref32, rtol=rt, atol=at)


# ------------------------------------------------------------------------------------------------ attention
@pytest.mark.parametrize("algo", list(ALGOS))
@pytest.mark.parametrize("name", list(G.ATTENTION_CASES))
def test_attention_forward_vs_golden(pkg, cuda_dev, golden, name, algo):
    cfg = G.ATTENTION_CASES[name]
    p = G.attention_inputs(cfg)
    m = _mk_attn(pkg, cfg, p, cuda_dev)
    m.algo = ALGOS[algo]
    x = p["x"].to(cuda_dev)
    with torch.no_grad():
        y = m(x, p["alpha"].to(cuda_dev)) if cfg["masked"] else m(x)
    _check_attention(y, p, cfg, algo, ref32=_t(golden["attention"][name + "/y"]))
    # dropped windows: bit-equal to the input (SURVEY.md section 4 property 2)
    if cfg["masked"]:
        keep = R.window_keep(p["alpha"], cfg["ws"], cfg["shift"])
        ws, s = cfg["ws"], cfg["shift"]
        ys = R.to_windows(torch.roll(y.cpu().permute(0, 2, 3, 1), (-s, -s), (1, 2)), ws)
        xs = R.to_windows(torch.roll(p["x"].permute(0, 2, 3, 1), (-s, -s), (1, 2)), ws)
        assert torch.equal(ys[~keep], xs[~keep])
        if bool(keep.any()):
            assert not torch.equal(ys[keep], xs[keep])


@pytest.mark.parametrize("algo", list(ALGOS))
@pytest.mark.parametrize("C,heads,ws,s,B,H,W,drop", [
    (192, 8, 8, 4, 2, 64, 96, 0.5),        # enc.attention1 / dec.attention2 geometry (scaled down)
    (80, 8, 4, 2, 2, 32, 48, 0.5),         # enc.attention2 / dec.attention1
    (192, 6, 8, 0, 1, 32, 32, 0.25),       # BASELINE config 4 (6 heads)
    (192, 6, 8, 4, 1, 32, 32, 0.75),
])
def test_attention_forward_vs_oracle_seeded(pkg, cuda_dev, C, heads, ws, s, B, H, W, drop, algo):
    cfg = dict(C=C, heads=heads, ws=ws, shift=s, B=B, H=H, W=W, drop=drop, masked=True, seed=100 + C + ws + s)
    p = G.attention_inputs(cfg)
    m = _mk_attn(pkg, cfg, p, cuda_dev)
    m.algo = ALGOS[algo]
    with torch.no_grad():
        y = m(p["x"].to(cuda_dev), p["alpha"].to(cuda_dev)).cpu()
        ycl = m(p["x"].to(cuda_dev).contiguous(memory_format=torch.channels_last), p["alpha"].to(cuda_dev))
    _check_attention(y, p, cfg, algo)
    assert ycl.is_contiguous(memory_format=torch.channels_last)
    _check_attention(ycl, p, cfg, algo)


@pytest.mark.parametrize("scale", [1.0, 3.0])
@pytest.mark.parametrize("C,heads,ws,s,B,H,W", [(192, 8, 8, 4, 2, 64, 96), (80, 8, 4, 2, 2, 32, 48),
                                                (192, 6, 8, 4, 1, 64, 64), (192, 8, 8, 4, 1, 24, 40)])
def test_attention_north_star_tolerance_at_random_init(pkg, cuda_dev, C, heads, ws, s, B, H, W, scale):
    """BASELINE.json: "identical synthetic inputs and identical random-init weights: fp32 outputs within 1e-3
    relative / 1e-4 absolute".  Module default init (what the reference builds), x ~ N(0, scale^2), 40 % of the windows
    transparent.  EVERY element of the default path's output meets the bound (and so does the forced SIMT kernel)."""
    torch.manual_seed(C + heads)
    m = pkg.MaskedWinBasedAttention(C, heads, ws, s)
    gen = torch.Generator().manual_seed(7)
    x = torch.randn(B, C, H, W, generator=gen) * scale
    alpha = G.blob_alpha(B, H, W, ws, s, 0.4, 99)
    a = m.attn
    ref = R.masked_window_attention(x.double(), alpha.double(), a.qkv.weight.detach().double(),
                                    a.qkv.bias.detach().double(), a.proj.weight.detach().double(),
                                    a.proj.bias.detach().double(), a.relative_position_bias_table.detach().double(),
                                    heads, ws, s)
    m = m.to(cuda_dev)
    with torch.no_grad():
        m.algo = ALGOS["simt"]
        y_simt = m(x.to(cuda_dev), alpha.to(cuda_dev)).cpu().double()
        m.algo = ALGOS["auto"]
        y_auto = m(x.to(cuda_dev), alpha.to(cuda_dev)).cpu().double()
        y_cl = m(x.to(cuda_dev).contiguous(memory_format=torch.channels_last), alpha.to(cuda_dev))
    torch.testing.assert_close(y_simt, ref, rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(y_auto, ref, rtol=RTOL, atol=ATOL)
    assert y_cl.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(y_cl.cpu().double(), y_auto)          # channels-last inputs take the same kernels


def test_alpha_one_equals_unmasked_bit_exact(pkg, cuda_dev):
    cfg = G.ATTENTION_CASES["attn_c192_h8_ws8_s4"]
    p = G.attention_inputs(cfg)
    m = _mk_attn(pkg, cfg, p, cuda_dev, masked=True)
    u = _mk_attn(pkg, cfg, p, cuda_dev, masked=False)
    x = p["x"].to(cuda_dev)
    with torch.no_grad():
        assert torch.equal(m(x, torch.ones(x.shape[0], 1, *x.shape[2:], device=cuda_dev)), u(x))


def test_attention_shape_errors(pkg, cuda_dev):
    m = pkg.MaskedWinBasedAttention(32, 4, 4, 2).to(cuda_dev)
    with pytest.raises(RuntimeError):
        m(torch.randn(1, 32, 10, 8, device=cuda_dev), torch.ones(1, 1, 10, 8, device=cuda_dev))


def test_attention_is_graph_capturable_and_counts_kept(pkg, cuda_dev, lib):
    cfg = G.ATTENTION_CASES["attn_c80_h8_ws4_s2"]
    p = G.attention_inputs(cfg)
    m = _mk_attn(pkg, cfg, p, cuda_dev)
    x, a = p["x"].to(cuda_dev), p["alpha"].to(cuda_dev)
    with torch.no_grad():
        eager = m(x, a)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):              # would raise on any host sync inside forward
            out = m(x, a)
        graph.replay()
        torch.cuda.synchronize()
    assert torch.equal(out, eager)
    kept = torch.zeros(1, dtype=torch.int32, device=cuda_dev)
    blk = m.attn._param_block(m.attn.qkv.weight, m.attn.qkv.bias, m.attn.proj.weight, m.attn.proj.bias,
                              m.attn.relative_position_bias_table)
    o2 = torch.empty_like(x)
    wsp = torch.empty(int(lib.mwa_workspace_bytes(x.shape[0], x.shape[2], x.shape[3], cfg["ws"])), dtype=torch.uint8,
                      device=cuda_dev)
    st = lib.mwa_forward(x.data_ptr(), a.data_ptr(), o2.data_ptr(), blk.data_ptr(), *x.shape, cfg["heads"], cfg["ws"],
                         cfg["shift"], 0, 0, kept.data_ptr(), wsp.data_ptr(), wsp.numel(),
                         torch.cuda.current_stream().cuda_stream)
    assert st == 0
    assert int(kept.item()) == int(R.window_keep(p["alpha"], cfg["ws"], cfg["shift"]).sum())


def test_window_attention_tokens_with_mask(pkg, cuda_dev):
    wa = pkg.WindowAttention(dim=32, window_size=(4, 4), num_heads=4).to(cuda_dev)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(6, 16, 32, generator=g)
    mask = torch.randn(3, 16, 16, generator=g)
    with torch.no_grad():
        wa.relative_position_bias_table.normal_(0, 0.5)
        y = wa(x.to(cuda_dev), mask.to(cuda_dev)).cpu()
        y0 = wa(x.to(cuda_dev)).cpu()
    args = [t.detach().cpu() for t in (wa.qkv.weight, wa.qkv.bias, wa.proj.weight, wa.proj.bias,
                                      wa.relative_position_bias_table)]
    torch.testing.assert_close(y, R.window_attention(x, *args, 4, 4, mask=mask.repeat(2, 1, 1)), rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(y0, R.window_attention(x, *args, 4, 4), rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("algo", list(ALGOS))
@pytest.mark.parametrize("name", list(G.ATTENTION_CASES))
def test_attention_backward_vs_golden(pkg, cuda_dev, golden, name, algo):
    """attention backward against the reference's autograd gradients: `simt` = the all-in-one mwa_backward kernel,
    `auto` = gather / core / scatter kernels around library token GEMMs.  Both are fp32 and re-compute from x, so the
    gradients do not depend on the precision of the forward kernel."""
    cfg = G.ATTENTION_CASES[name]
    p = G.attention_inputs(cfg)
    m = _mk_attn(pkg, cfg, p, cuda_dev)
    m.algo = ALGOS[algo]
    x = p["x"].to(cuda_dev).requires_grad_(True)
    y = m(x, p["alpha"].to(cuda_dev)) if cfg["masked"] else m(x)
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(cfg["seed"] + 5)).to(cuda_dev)
    y.backward(gy)
    g = golden["attention"]
    torch.testing.assert_close(x.grad.cpu(), _t(g[name + "/dx"]), rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(m.attn.relative_position_bias_table.grad.cpu(), _t(g[name + "/dtable"]), rtol=1e-3,
                               atol=1e-3)
    if name + "/dqkv_w" in g:
        torch.testing.assert_close(m.attn.qkv.weight.grad.cpu(), _t(g[name + "/dqkv_w"]), rtol=1e-3, atol=1e-3)
        torch.testing.assert_close(m.attn.proj.weight.grad.cpu(), _t(g[name + "/dproj_w"]), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("algo", list(ALGOS))
@pytest.mark.parametrize("channels_last", [False, True])
@pytest.mark.parametrize("name", ["attn_c80_h8_ws4_s2", "attn_c192_h8_ws8_s4"])
def test_attention_backward_all_gradients(pkg, cuda_dev, name, channels_last, algo):
    """every gradient (incl. the two bias vectors, which the golden file does not carry) against autograd through the
    oracle's fp64 re-statement; NHWC input gives the same gradients."""
    cfg = G.ATTENTION_CASES[name]
    p = G.attention_inputs(cfg)
    m = _mk_attn(pkg, cfg, p, cuda_dev)
    m.algo = ALGOS[algo]
    x = p["x"].to(cuda_dev)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    y = m(x, p["alpha"].to(cuda_dev))
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(3))
    y.backward(gy.to(cuda_dev))
    leaves = {k: (None if v is None else v.double().requires_grad_(k != "alpha")) for k, v in p.items()}
    ref = R.masked_window_attention(leaves["x"], leaves["alpha"], leaves["qkv_w"], leaves["qkv_b"], leaves["proj_w"],
                                    leaves["proj_b"], leaves["table"], cfg["heads"], cfg["ws"], cfg["shift"])
    ref.backward(gy.double())
    got = dict(x=x.grad, qkv_w=m.attn.qkv.weight.grad, qkv_b=m.attn.qkv.bias.grad, proj_w=m.attn.proj.weight.grad,
               proj_b=m.attn.proj.bias.grad, table=m.attn.relative_position_bias_table.grad)
    for k, v in got.items():
        torch.testing.assert_close(v.double().cpu(), leaves[k].grad, rtol=1e-3, atol=2e-4, msg=lambda s_, k=k: f"{k}: {s_}")


@pytest.mark.parametrize("algo", list(ALGOS))
def test_window_attention_tokens_backward(pkg, cuda_dev, algo):
    """window_attention_backward / mwa_bwd_core in token mode: WindowAttention.forward(x, mask) on pre-partitioned
    tokens."""
    wa = pkg.WindowAttention(dim=32, window_size=(4, 4), num_heads=4).to(cuda_dev)
    wa.algo = ALGOS[algo]
    g = torch.Generator().manual_seed(9)
    x = torch.randn(6, 16, 32, generator=g)
    mask = torch.randn(3, 16, 16, generator=g)
    gy = torch.randn(6, 16, 32, generator=g)
    with torch.no_grad():
        wa.relative_position_bias_table.normal_(0, 0.5)
    xd = x.to(cuda_dev).requires_grad_(True)
    wa(xd, mask.to(cuda_dev)).backward(gy.to(cuda_dev))
    names = ("qkv.weight", "qkv.bias", "proj.weight", "proj.bias", "relative_position_bias_table")
    params = [dict(wa.named_parameters())[n] for n in names]
    ref_leaves = [t.detach().double().cpu().requires_grad_(True) for t in params]
    xr = x.double().requires_grad_(True)
    R.window_attention(xr, *ref_leaves, 4, 4, mask=mask.double().repeat(2, 1, 1)).backward(gy.double())
    torch.testing.assert_close(xd.grad.double().cpu(), xr.grad, rtol=1e-3, atol=1e-4)
    for n, t, r in zip(names, params, ref_leaves):
        torch.testing.assert_close(t.grad.double().cpu(), r.grad, rtol=1e-3, atol=2e-4, msg=lambda s_, n=n: f"{n}: {s_}")


# ------------------------------------------------------------------------------------------------ GDN
@pytest.mark.parametrize("algo", list(ALGOS))
@pytest.mark.parametrize("name", list(G.GDN_CASES))
def test_gdn_forward_backward_vs_golden(pkg, cuda_dev, golden, name, algo):
    cfg = G.GDN_CASES[name]
    p = G.gdn_inputs(cfg)
    m = pkg.GDN(cfg["C"], inverse=cfg["inverse"])
    with torch.no_grad():
        m.beta.copy_(p["beta"])
        m.gamma.copy_(p["gamma"])
    m = m.to(cuda_dev)
    m.algo = ALGOS[algo]
    x = p["x"].to(cuda_dev).requires_grad_(True)
    y = m(x)
    g = golden["gdn"]
    assert y.shape == p["x"].shape
    if algo == "simt":
        torch.testing.assert_close(y.detach().cpu(), _t(g[name + "/y"]), rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(y.detach().cpu(), _t(g[name + "/y"]), rtol=RTOL, atol=ATOL)
    gy = torch.randn(y.shape, generator=torch.Generator().manual_seed(cfg["seed"] + 5)).to(cuda_dev)
    y.backward(gy)
    torch.testing.assert_close(x.grad.cpu(), _t(g[name + "/dx"]), rtol=1e-3, atol=1e-4)
    torch.testing.assert_close(m.beta.grad.cpu(), _t(g[name + "/dbeta"]), rtol=1e-3, atol=1e-3)
    torch.testing.assert_close(m.gamma.grad.cpu(), _t(g[name + "/dgamma"]), rtol=1e-3, atol=1e-3)


@pytest.mark.parametrize("algo", list(ALGOS))
@pytest.mark.parametrize("inverse", [False, True])
@pytest.mark.parametrize("B,H,W", [(2, 64, 96), (1, 37, 53), (3, 8, 12)])
def test_gdn_forward_vs_oracle_seeded(pkg, cuda_dev, inverse, B, H, W, algo):
    cfg = dict(C=192, B=B, H=H, W=W, inverse=inverse, seed=200 + H)
    p = G.gdn_inputs(cfg)
    m = pkg.GDN(192, inverse=inverse)
    with torch.no_grad():
        m.beta.copy_(p["beta"])
        m.gamma.copy_(p["gamma"])
    m = m.to(cuda_dev)
    m.algo = ALGOS[algo]
    ref = R.gdn(p["x"].double(), p["beta"].double(), p["gamma"].double(), inverse=inverse)
    with torch.no_grad():
        y = m(p["x"].to(cuda_dev))
        ycl = m(p["x"].to(cuda_dev).contiguous(memory_format=torch.channels_last))
    torch.testing.assert_close(y.cpu().double(), ref, rtol=RTOL, atol=ATOL)
    torch.testing.assert_close(ycl.cpu().double(), ref, rtol=RTOL, atol=ATOL)
    assert ycl.is_contiguous(memory_format=torch.channels_last)


def test_gdn_param_block_follows_parameter_updates(pkg, cuda_dev):
    m = pkg.GDN(16).to(cuda_dev)
    x = torch.randn(1, 16, 8, 8, device=cuda_dev)
    with torch.no_grad():
        y0 = m(x)
        m.beta.mul_(2.0)                       # in-place update bumps _version -> block rebuilt
        y1 = m(x)
    assert not torch.equal(y0, y1)
    ref = R.gdn(x.cpu(), m.beta.detach().cpu(), m.gamma.detach().cpu())
    torch.testing.assert_close(y1.cpu(), ref, rtol=2e-5, atol=2e-6)


# ------------------------------------------------------------------------------------------------ rounding
def test_rounding_bit_exact_vs_golden(pkg, cuda_dev, golden):
    p = {k: v.to(cuda_dev) for k, v in G.rounding_inputs().items()}
    g = golden["rounding"]
    assert np.array_equal(pkg.ste_round(p["x"]).cpu().numpy(), g["ste_round"])
    assert np.array_equal(pkg.quantize_offset(p["x"], p["mu"]).cpu().numpy(), g["quantize_offset"])
    assert np.array_equal(pkg.quantize_levels(p["m"], 255).cpu().numpy(), g["levels255"])
    np.testing.assert_allclose(pkg.lrp_add(p["x"], p["lrp"]).cpu().numpy(), g["lrp_add"], rtol=1e-6, atol=1e-6)
    # signed zero of round-half-even is preserved (-0.5 -> -0.0)
    assert np.array_equal(np.signbit(pkg.ste_round(p["x"]).cpu().numpy()), np.signbit(g["ste_round"]))


def test_rounding_on_channel_chunks_and_channel_offsets(pkg, cuda_dev):
    g = torch.Generator().manual_seed(7)
    y = (torch.randn(3, 80, 6, 10, generator=g) * 4).to(cuda_dev)
    mu = torch.randn(3, 8, 6, 10, generator=g).to(cuda_dev)
    for i, ys in enumerate(y.chunk(10, 1)):                    # non-contiguous views, consumed in place
        out = pkg.quantize_offset(ys, mu)
        assert torch.equal(out, torch.round(ys - mu) + mu)
        assert torch.equal(pkg.ste_round(ys), torch.round(ys))
    med = torch.randn(1, 80, 1, 1, generator=g).to(cuda_dev)
    assert torch.equal(pkg.quantize_offset(y, med), torch.round(y - med) + med)
    odd = (torch.randn(1001, generator=g) * 3).to(cuda_dev)[1:]   # misaligned pointer -> scalar path
    assert torch.equal(pkg.ste_round(odd), torch.round(odd))
    assert pkg.ste_round(torch.empty(0, device=cuda_dev)).numel() == 0


def test_rounding_gradients(pkg, cuda_dev):
    x = torch.randn(64, device=cuda_dev, requires_grad=True)
    mu = torch.randn(64, device=cuda_dev, requires_grad=True)
    lrp = torch.randn(64, device=cuda_dev, requires_grad=True)
    out = pkg.lrp_add(pkg.quantize_offset(x, mu), lrp)
    out.backward(torch.ones_like(out))
    assert torch.equal(x.grad, torch.ones_like(x))             # straight-through
    assert torch.equal(mu.grad, torch.zeros_like(mu))
    torch.testing.assert_close(lrp.grad, 0.5 * (1 - torch.tanh(lrp.detach()) ** 2))
