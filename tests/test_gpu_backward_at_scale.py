"""The training backward at the sizes training runs it (BASELINE config 5: 8 crops of 256^2 -> 512 windows of 8x8, 32,768
tokens in enc.attention1 / dec.attention2), against plain fp64 CPU references.

  A. gemm_tokens_forward -- the tcgen05 token GEMM of the attention backward (conv_split_cl_kernel, conv_prepare kind 0 / 2
     at k = 1, conv_tc_kernel<192, true> with its token-major epilogue, the in_scale gradient pre-scaling).  conv.gemm_tokens
     only launches it for GEMMs of at least GEMM_TOKENS_MIN_FLOP; the tests lower that threshold to 0 and check through a
     spy on the library entry point that the kernel ran.  The bound is per element and relative to |x| |W|^T + |b|: at
     gradient magnitudes (~1e-7) any fixed absolute tolerance would accept a kernel that is plain fp16.  Bound 2e-6;
     observed on an NVIDIA B200 (1000 W power limit): at most 7.6e-7 (T = 32,768, Cin 192, Cout 576), against ~1.3e-4
     for a kernel that drops one of its three passes (emulated on the CPU, O(1) activations).
  B. the default (gather / core / scatter) attention backward at training size and the default threshold, with real
     gradient magnitudes (grad_out ~ 2^-20), including scale equivariance and a negative control without the input scaling.
  C. the GDN backward: the GEMM-composed path (AUTO) and the SIMT kernel, NCHW and channels-last, above 96 pixels.

Tolerances scale with the data (the reference's magnitude or the grad_out scale), never a fixed absolute number.  The
observed maxima of every check are attached to the test report (`record_property`: pytest --junitxml shows them).
"""
import functools

import pytest
import torch

from oracle import golden_cases as G
from oracle import ref_ops as R

pytestmark = pytest.mark.gpu

MWA_OK, MWA_ERR_UNSUPPORTED, MWA_ERR_ALIGNMENT = 0, -2, -3
ALGO_AUTO, ALGO_SIMT = 0, 1


class _Spy:
    """wraps one C entry point of the library for the duration of a test and records (args, status) of every call"""

    def __init__(self, monkeypatch, lib, name):
        real = getattr(lib, name)
        self.calls = []

        def spy(*args):
            st = real(*args)
            self.calls.append((args, st))
            return st

        monkeypatch.setattr(lib, name, spy)


def _max_rel(got, ref):
    """max |got - ref| / max |ref| (both fp64 CPU)"""
    return float((got - ref).abs().max()) / max(float(ref.abs().max()), 1e-300)


# ================================================================================================ A. token GEMM kernel
GEMM_BOUND = 2e-6          # per element, relative to |x| |W|^T + |b|

GEMM_SHAPES = {
    # (T, Cin, Cout)
    "qkv_c192": (4096, 192, 576),          # three 192-column N blocks
    "dao_c192": (4096, 192, 192),
    "dxw_c192": (4096, 576, 192),          # nine K blocks: several tensor-core chunks per tile
    "qkv_c80": (4096, 80, 240),            # two N blocks of 128, padded to 256
    "dao_c80": (4096, 80, 80),
    "dxw_c80": (4096, 240, 80),
    "cout8": (4096, 192, 8),
    "cin20": (4096, 20, 64),               # K padded to 24 (split planes) and to 32 (MMA)
    "cin120": (4096, 120, 240),            # a partial second K block
    "t32": (32, 192, 576),                 # one row of the 32-wide token image
    "t224": (32 * 7, 192, 192),            # 7 rows: the last 4-row tile is partial
    "t4128": (32 * 129, 80, 240),          # 129 rows: the last tile has one row
    "t32768": (32768, 192, 576),           # config 5: more tiles than SMs, grid-stride split kernel
}


def _tokens(T, cin, kind, gen):
    """(T, Cin) fp32 CPU input of one magnitude class, and whether gemm_tokens should pre-scale it"""
    if kind == "act":
        return torch.randn(T, cin, generator=gen) * 1.5, False
    if kind == "act1e4":           # well inside the +-1.3e5 range of fp16 hi + lo
        return torch.randn(T, cin, generator=gen) * 1e4, False
    if kind == "grad1e-7":
        return torch.randn(T, cin, generator=gen) * 1e-7, True
    if kind == "grad1e-12":
        return torch.randn(T, cin, generator=gen) * 1e-12, True
    if kind == "dropped":          # gradients with the all-zero 64-token blocks of dropped windows
        x = torch.randn(T, cin, generator=gen) * 1e-7
        keep = (torch.rand(max(T // 64, 1), generator=gen) >= 0.4).repeat_interleave(64)[:T]
        x[~keep] = 0.0
        return x, True
    raise ValueError(kind)


def _run_gemm(pkg, dev, x, w, b, in_out, scale):
    """conv.gemm_tokens on the GPU: out = x W^T + b with W (Cout, Cin), passed as (Cin, Cout) when in_out"""
    wd = (w.t().contiguous() if in_out else w).to(dev)
    out = pkg.conv.gemm_tokens(x.to(dev), wd, None if b is None else b.to(dev), weight_is_in_out=in_out,
                               scale_input=scale)
    torch.cuda.synchronize()
    return out.cpu().double()


def _gemm_ratio(out, x, w, b):
    """max over elements of |out - ref| / (|x| |W|^T + |b|); an error where that is 0 counts as infinite.  In row
    blocks, to keep the fp64 working set small."""
    w64 = w.double()
    worst = 0.0
    for r0 in range(0, x.shape[0], 4096):
        x64 = x[r0:r0 + 4096].double()
        ref = x64 @ w64.t()
        den = x64.abs() @ w64.abs().t()
        if b is not None:
            ref += b.double()
            den += b.double().abs()
        err = (out[r0:r0 + 4096] - ref).abs()
        if bool((err[den == 0] > 0).any()):
            return float("inf")
        worst = max(worst, float((err / den.clamp_min(1e-300)).max()))
    return worst


def _check_kernel_calls(spy, expect):
    """spy saw exactly the (T, Cin, Cout) calls in `expect`, each returning MWA_OK"""
    got = [(int(a[1]), int(a[2]), int(a[5])) for a, _ in spy.calls]
    assert got == expect, f"gemm_tokens_forward calls {got}, expected {expect}"
    assert all(st == MWA_OK for _, st in spy.calls)


@pytest.fixture
def gemm_spy(monkeypatch, lib):
    return _Spy(monkeypatch, lib, "gemm_tokens_forward")


@pytest.mark.parametrize("in_out", [False, True], ids=["w_out_in", "w_in_out"])
@pytest.mark.parametrize("name", list(GEMM_SHAPES))
def test_gemm_tokens_shapes_vs_fp64(cuda_dev, pkg, gemm_spy, monkeypatch, record_property, name, in_out):
    """O(1) activations with a bias at every shape: the real token GEMMs of both attention layers and the edges of the
    kernel's tiling (Cout = 8, Cin padded, partial and single tiles, grid-stride).  in_out selects the image kind
    (0: W given (Cout, Cin); 2: W given (Cin, Cout), the dao / dxw GEMMs)."""
    monkeypatch.setattr(pkg.conv, "GEMM_TOKENS_MIN_FLOP", 0)
    T, cin, cout = GEMM_SHAPES[name]
    gen = torch.Generator().manual_seed(T + 7 * cin + cout)
    x, _ = _tokens(T, cin, "act", gen)
    w = torch.randn(cout, cin, generator=gen) * cin ** -0.5
    b = torch.randn(cout, generator=gen) * 0.5
    out = _run_gemm(pkg, cuda_dev, x, w, b, in_out, False)
    _check_kernel_calls(gemm_spy, [(T, cin, cout)])
    r = _gemm_ratio(out, x, w, b)
    record_property("max_err_over_absprod", r)
    assert r <= GEMM_BOUND, f"max |err| / (|x||W|^T + |b|) = {r:.3e} > {GEMM_BOUND}"


@pytest.mark.parametrize("bias", [False, True], ids=["nobias", "bias"])
@pytest.mark.parametrize("in_out", [False, True], ids=["w_out_in", "w_in_out"])
@pytest.mark.parametrize("kind", ["act", "act1e4", "grad1e-7", "grad1e-12", "dropped"])
@pytest.mark.parametrize("name", ["qkv_c192", "dxw_c192", "qkv_c80"])
def test_gemm_tokens_value_ranges_vs_fp64(cuda_dev, pkg, gemm_spy, monkeypatch, record_property, name, kind, in_out,
                                          bias):
    """activations of O(1) and ~1e4 as they are; gradients of ~1e-7 and ~1e-12 (and ones with the zero rows of dropped
    windows) pre-scaled by conv.gradient_scale.  The bias is of the output's magnitude, so a bias that were divided by
    the input scale -- or scaled at all -- would be far outside the bound."""
    monkeypatch.setattr(pkg.conv, "GEMM_TOKENS_MIN_FLOP", 0)
    T, cin, cout = GEMM_SHAPES[name]
    gen = torch.Generator().manual_seed(3 * T + cin + cout + len(kind))
    x, scale = _tokens(T, cin, kind, gen)
    w = torch.randn(cout, cin, generator=gen) * cin ** -0.5
    b = torch.randn(cout, generator=gen) * float(x.std()) if bias else None
    out = _run_gemm(pkg, cuda_dev, x, w, b, in_out, scale)
    _check_kernel_calls(gemm_spy, [(T, cin, cout)])
    assert bool(torch.isfinite(out).all())
    r = _gemm_ratio(out, x, w, b)
    record_property("max_err_over_absprod", r)
    assert r <= GEMM_BOUND, f"max |err| / (|x||W|^T + |b|) = {r:.3e} > {GEMM_BOUND}"


@pytest.mark.parametrize("bias", [False, True], ids=["nobias", "bias"])
def test_gemm_tokens_zero_input_with_scale(cuda_dev, pkg, gemm_spy, monkeypatch, bias):
    """an all-zero gradient (every window dropped) gets the largest input scale gradient_scale can produce (2^109): the
    result is exactly the bias, finite, with no 0 * inf or overflow anywhere"""
    monkeypatch.setattr(pkg.conv, "GEMM_TOKENS_MIN_FLOP", 0)
    T, cin, cout = GEMM_SHAPES["dxw_c192"]
    gen = torch.Generator().manual_seed(5)
    w = torch.randn(cout, cin, generator=gen) * cin ** -0.5
    b = torch.randn(cout, generator=gen) if bias else None
    out = _run_gemm(pkg, cuda_dev, torch.zeros(T, cin), w, b, True, True)
    _check_kernel_calls(gemm_spy, [(T, cin, cout)])
    assert bool(torch.isfinite(out).all())
    want = torch.zeros(T, cout, dtype=torch.float64) if b is None else b.double().expand(T, cout)
    assert torch.equal(out, want)


def test_gemm_tokens_abi_contract(cuda_dev, lib):
    """status codes of gemm_tokens_forward on real device buffers"""
    T, cin, cout = 64, 192, 192
    dev = cuda_dev
    st = torch.cuda.current_stream().cuda_stream
    w = torch.randn(cout, cin, device=dev)
    nbytes = int(lib.conv_image_bytes(0, cin, cout, 1, 1))
    img = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    assert lib.conv_prepare(w.data_ptr(), 0, cin, cout, 1, 1, img.data_ptr(), nbytes, st) == MWA_OK
    xbuf = torch.randn(T * cin + 4, device=dev)
    x = xbuf[:T * cin]
    split = torch.empty(2, (T + 32) * cin, dtype=torch.int16, device=dev)
    out = torch.full((T + 32, cout + 8), 7.0, device=dev)

    def call(xp, t, co):
        return lib.gemm_tokens_forward(xp, t, cin, None, out.data_ptr(), co, img.data_ptr(), split[0].data_ptr(),
                                       split[1].data_ptr(), None, st)

    assert call(x.data_ptr(), T + 16, cout) == MWA_ERR_UNSUPPORTED          # T % 32 != 0
    assert call(x.data_ptr(), T, cout - 4) == MWA_ERR_UNSUPPORTED           # Cout % 8 != 0
    assert call(x.data_ptr(), 0, cout) == MWA_OK                            # nothing to do
    assert call(xbuf[1:].data_ptr(), T, cout) == MWA_ERR_ALIGNMENT          # x 4 bytes off a 16-byte boundary
    torch.cuda.synchronize()
    assert bool((out == 7.0).all())                                         # no call above wrote anything
    assert call(x.data_ptr(), T, cout) == MWA_OK
    torch.cuda.synchronize()
    ref = x.view(T, cin).double() @ w.double().t()
    got = out.view(-1)[:T * cout].view(T, cout).double()
    den = x.view(T, cin).double().abs() @ w.double().abs().t()
    assert float(((got - ref).abs() / den).max()) <= GEMM_BOUND


# ================================================================================================ B. attention backward
GRAD_SCALE = 2.0 ** -20         # the magnitude of real loss gradients at this point of the model
ATTN_BOUND = 2e-5               # max |err| <= ATTN_BOUND * max |ref|, per gradient (B200: at most 4.6e-6, grad x)
GRAD_NAMES = ("x", "qkv_w", "qkv_b", "proj_w", "proj_b", "table")
# The weight and bias gradients are sums over every token (32,768 - 65,536 here, up to ~1.5e3 for grad_out ~ N(0, 1)).
# The small-size tests' absolute floor of 2e-4 is ~1e-7 of such a sum, below what fp32 accumulation delivers at this
# length: against fp64, the oracle itself evaluated in fp32 on the CPU has 39 elements of dWqkv beyond 1e-3 |ref| + 2e-4 at
# 512 windows, and this backward fed with correctly rounded fp32 token GEMMs has 26 (NVIDIA B200).  Their absolute floor
# scales with the sum instead, like GDN's dbeta / dgamma below: 1e-5 max |ref|.
TOKEN_SUMS = ("qkv_w", "qkv_b", "proj_w", "proj_b")

ATTN_CASES = {
    # name: (C, heads, ws, shift, B, H, W), token-GEMM kernel calls per backward at the default threshold
    "c192_h8_b8_64x64": ((192, 8, 8, 4, 8, 64, 64), 3),       # config 5 enc.attention1: 512 windows, 32,768 tokens
    "c192_h6_b4_96x96": ((192, 6, 8, 4, 4, 96, 96), 3),       # 576 windows
    "c80_h8_b4_128x128": ((80, 8, 4, 2, 4, 128, 128), 2),     # 4,096 windows: dao (0.84 GFLOP) stays on the library
}


def _attn_cfg(name):
    (C, heads, ws, shift, B, H, W), _ = ATTN_CASES[name]
    return dict(C=C, heads=heads, ws=ws, shift=shift, B=B, H=H, W=W, drop=0.4, masked=True, seed=400 + C + H)


@functools.lru_cache(maxsize=1)
def _attn_reference(name):
    """inputs (G.attention_inputs: ~40 % of the windows dropped through G.blob_alpha), grad_out ~ N(0, 1), and the six
    gradients of fp64 autograd through the oracle for that grad_out.  One image at a time (windows never cross images),
    so the CPU working set stays a few hundred MB."""
    cfg = _attn_cfg(name)
    p = G.attention_inputs(cfg)
    gy = torch.randn(p["x"].shape, generator=torch.Generator().manual_seed(cfg["seed"] + 1))
    params = {k: p[k].double().requires_grad_(True) for k in GRAD_NAMES[1:]}
    gx = []
    for b in range(cfg["B"]):
        xb = p["x"][b:b + 1].double().requires_grad_(True)
        y = R.masked_window_attention(xb, p["alpha"][b:b + 1].double(), params["qkv_w"], params["qkv_b"],
                                      params["proj_w"], params["proj_b"], params["table"], cfg["heads"], cfg["ws"],
                                      cfg["shift"])
        y.backward(gy[b:b + 1].double())
        gx.append(xb.grad)
    ref = {"x": torch.cat(gx)}
    ref.update({k: v.grad for k, v in params.items()})
    return p, gy, ref


def _mk_attn(pkg, cfg, p, dev):
    m = pkg.MaskedWinBasedAttention(dim=cfg["C"], num_heads=cfg["heads"], window_size=cfg["ws"], shift_size=cfg["shift"])
    with torch.no_grad():
        m.attn.qkv.weight.copy_(p["qkv_w"])
        m.attn.qkv.bias.copy_(p["qkv_b"])
        m.attn.proj.weight.copy_(p["proj_w"])
        m.attn.proj.bias.copy_(p["proj_b"])
        m.attn.relative_position_bias_table.copy_(p["table"])
    return m.to(dev)


def _attn_grads(m, x):
    a = m.attn
    g = dict(x=x.grad, qkv_w=a.qkv.weight.grad, qkv_b=a.qkv.bias.grad, proj_w=a.proj.weight.grad,
             proj_b=a.proj.bias.grad, table=a.relative_position_bias_table.grad)
    return {k: v.detach().cpu().double() for k, v in g.items()}


def _attn_backward(pkg, dev, name, channels_last, scales):
    """GPU forward once, then one backward per grad_out scale; returns the per-scale gradients and kernel calls"""
    cfg = _attn_cfg(name)
    p, gy, _ = _attn_reference(name)
    m = _mk_attn(pkg, cfg, p, dev)
    x = p["x"].to(dev)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    y = m(x, p["alpha"].to(dev))
    gyd = gy.to(dev)
    lib = pkg._abi.load()
    out = []
    for i, s in enumerate(scales):
        x.grad = None
        m.zero_grad(set_to_none=True)
        with pytest.MonkeyPatch.context() as mp:
            spy = _Spy(mp, lib, "gemm_tokens_forward")
            y.backward(gyd * s, retain_graph=i + 1 < len(scales))
            torch.cuda.synchronize()
        out.append((_attn_grads(m, x), spy.calls))
    return out


def _expected_calls(pkg, name):
    """the token GEMMs of one backward that reach conv.GEMM_TOKENS_MIN_FLOP, in launch order: qkv, dao, dxw"""
    (C, _, _, _, B, H, W), n = ATTN_CASES[name]
    T = B * H * W
    want = [c for c in ((T, C, 3 * C), (T, C, C), (T, 3 * C, C)) if 2.0 * c[0] * c[1] * c[2] >= pkg.conv.GEMM_TOKENS_MIN_FLOP]
    assert len(want) == n
    return want


@pytest.mark.parametrize("name,channels_last", [("c192_h8_b8_64x64", False), ("c192_h8_b8_64x64", True),
                                                ("c192_h6_b4_96x96", False), ("c80_h8_b4_128x128", False)])
def test_attention_backward_at_training_size(cuda_dev, pkg, record_property, name, channels_last):
    """All six gradients of the default attention backward at training size against fp64 autograd, grad_out =
    N(0, 1) * 2^-20: the suite's all-gradients tolerance scaled by 2^-20 (rtol 1e-3, atol 2e-4 * 2^-20; for the
    token sums in TOKEN_SUMS atol 1e-5 max |ref|), and max |err| <= 2e-5 max |ref| per gradient.  Then grad_out * 2^-24:
    every stage is fp32 arithmetic linear in grad_out with power-of-two input scaling, so the gradients are bit-identical
    after multiplying back by 2^4 -- except the relative-position table's, which is accumulated with atomics (1e-6
    relative)."""
    _, _, ref = _attn_reference(name)
    (g20, calls20), (g24, calls24) = _attn_backward(pkg, cuda_dev, name, channels_last, (GRAD_SCALE, GRAD_SCALE / 16))
    want = _expected_calls(pkg, name)
    for calls in (calls20, calls24):
        got = [(int(a[1]), int(a[2]), int(a[5])) for a, _ in calls]
        assert got == want, f"token-GEMM kernel calls {got}, expected {want}"
        assert all(st == MWA_OK for _, st in calls)
    rel = {k: _max_rel(g20[k], ref[k] * GRAD_SCALE) for k in GRAD_NAMES}
    exact = {k: torch.equal(g24[k] * 16, g20[k]) for k in GRAD_NAMES if k != "table"}
    table_rel = _max_rel(g24["table"] * 16, g20["table"])
    for k, v in rel.items():
        record_property(f"max_err_over_max_ref_{k}", v)
    record_property("equivariant_bit_exact", all(exact.values()))
    record_property("equivariance_table_rel", table_rel)
    failed = []
    for k in GRAD_NAMES:
        r = ref[k] * GRAD_SCALE
        atol = 1e-5 * float(r.abs().max()) if k in TOKEN_SUMS else 2e-4 * GRAD_SCALE
        try:
            torch.testing.assert_close(g20[k], r, rtol=1e-3, atol=atol)
        except AssertionError as e:
            failed.append(f"{k}: {e}")
        if rel[k] > ATTN_BOUND:
            failed.append(f"{k}: max |err| / max |ref| = {rel[k]:.3e} > {ATTN_BOUND}")
    if not all(exact.values()):
        failed.append(f"not bit-identical after x 2^4: {[k for k, v in exact.items() if not v]}")
    if table_rel > 1e-6:
        failed.append(f"table gradient after x 2^4: {table_rel:.3e} relative")
    assert not failed, "\n".join(failed) + f"\nmax |err| / max |ref|: {rel}"


def test_attention_backward_needs_gradient_scaling(cuda_dev, pkg, monkeypatch, record_property):
    """negative control: with conv.gradient_scale pinned to 1 the token GEMMs split ~1e-6 gradients into fp16 as they
    are (subnormal there) and the 2^-20 case of the test above falls outside its bound -- that test depends on the
    input scaling"""
    monkeypatch.setattr(pkg.conv, "gradient_scale", lambda g: torch.ones(1, device=g.device))
    name = "c80_h8_b4_128x128"
    _, _, ref = _attn_reference(name)
    ((g20, calls),) = _attn_backward(pkg, cuda_dev, name, False, (GRAD_SCALE,))
    assert len(calls) == 2
    rel = {k: _max_rel(g20[k], ref[k] * GRAD_SCALE) for k in GRAD_NAMES}
    for k, v in rel.items():
        record_property(f"unscaled_max_err_over_max_ref_{k}", v)
    assert rel["x"] > ATTN_BOUND, rel


def test_window_attention_tokens_backward_on_kernel(cuda_dev, pkg, lib, monkeypatch):
    """WindowAttention.forward(x, mask) (token mode of mwa_bwd_core) with all three token GEMMs on the kernel"""
    monkeypatch.setattr(pkg.conv, "GEMM_TOKENS_MIN_FLOP", 0)
    spy = _Spy(monkeypatch, lib, "gemm_tokens_forward")
    wa = pkg.WindowAttention(dim=32, window_size=(4, 4), num_heads=4).to(cuda_dev)
    g = torch.Generator().manual_seed(9)
    x = torch.randn(6, 16, 32, generator=g)
    mask = torch.randn(3, 16, 16, generator=g)
    gy = torch.randn(6, 16, 32, generator=g)
    with torch.no_grad():
        wa.relative_position_bias_table.normal_(0, 0.5)
    xd = x.to(cuda_dev).requires_grad_(True)
    wa(xd, mask.to(cuda_dev)).backward(gy.to(cuda_dev))
    _check_kernel_calls(spy, [(96, 32, 96), (96, 32, 32), (96, 96, 32)])
    names = ("qkv.weight", "qkv.bias", "proj.weight", "proj.bias", "relative_position_bias_table")
    params = [dict(wa.named_parameters())[n] for n in names]
    ref_leaves = [t.detach().double().cpu().requires_grad_(True) for t in params]
    xr = x.double().requires_grad_(True)
    R.window_attention(xr, *ref_leaves, 4, 4, mask=mask.double().repeat(2, 1, 1)).backward(gy.double())
    torch.testing.assert_close(xd.grad.double().cpu(), xr.grad, rtol=1e-3, atol=1e-4)
    for n, t, r in zip(names, params, ref_leaves):
        torch.testing.assert_close(t.grad.double().cpu(), r.grad, rtol=1e-3, atol=2e-4, msg=lambda s_, n=n: f"{n}: {s_}")


# ================================================================================================ C. GDN backward
GDN_SHAPES = {"2x192x128x128": (2, 192, 128, 128), "1x192x37x53": (1, 192, 37, 53)}


@functools.lru_cache(maxsize=1)
def _gdn_reference(shape, inverse, hit_bounds=False):
    """G.gdn_inputs' construction (beta, gamma away from their initial values; hit_bounds: entries below the bounds),
    grad_out ~ N(0, 1), and the fp64 autograd gradients of R.gdn (LowerBound's pass-through rule included)"""
    B, C, H, W = shape
    p = G.gdn_inputs(dict(C=C, B=B, H=H, W=W, seed=500 + C + H, hit_bounds=hit_bounds))
    gy = torch.randn(shape, generator=torch.Generator().manual_seed(600 + H))
    leaves = {k: p[k].double().requires_grad_(True) for k in ("x", "beta", "gamma")}
    R.gdn(leaves["x"], leaves["beta"], leaves["gamma"], inverse=inverse).backward(gy.double())
    return p, gy, {k: v.grad for k, v in leaves.items()}


def _gdn_backward(pkg, lib, dev, p, gy, inverse, algo, channels_last):
    """GPU GDN forward + backward; returns the gradients and which backward ran ("composed" or "simt")"""
    C = p["beta"].shape[0]
    m = pkg.GDN(C, inverse=inverse)
    with torch.no_grad():
        m.beta.copy_(p["beta"])
        m.gamma.copy_(p["gamma"])
    m = m.to(dev)
    m.algo = algo
    x = p["x"].to(dev)
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    with pytest.MonkeyPatch.context() as mp:
        simt, composed = _Spy(mp, lib, "gdn_backward"), _Spy(mp, lib, "gdn_bwd_dn")
        m(x).backward(gy.to(dev))
        torch.cuda.synchronize()
    assert len(simt.calls) + len(composed.calls) == 1
    path = "simt" if simt.calls else "composed"
    if composed.calls:
        assert int(composed.calls[0][0][9]) == int(channels_last)       # the layout the composed stages were told
    grads = dict(x=x.grad, beta=m.beta.grad, gamma=m.gamma.grad)
    return {k: v.detach().cpu().double() for k, v in grads.items()}, path


def _check_gdn(got, ref, record_property):
    rel = {k: _max_rel(got[k], ref[k]) for k in ("x", "beta", "gamma")}
    for k, v in rel.items():
        record_property(f"max_err_over_max_ref_{k}", v)
    torch.testing.assert_close(got["x"], ref["x"], rtol=1e-3, atol=1e-4)
    for k in ("beta", "gamma"):          # sums over every pixel
        torch.testing.assert_close(got[k], ref[k], rtol=1e-3, atol=1e-5 * float(ref[k].abs().max()),
                                   msg=lambda s_, k=k: f"d{k}: {s_}")


@pytest.mark.parametrize("algo", [ALGO_AUTO, ALGO_SIMT], ids=["auto", "simt"])
@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("inverse", [False, True], ids=["gdn", "igdn"])
@pytest.mark.parametrize("shape", list(GDN_SHAPES))
def test_gdn_backward_vs_fp64(cuda_dev, pkg, lib, record_property, shape, inverse, channels_last, algo):
    """dx, dbeta, dgamma of GDN / IGDN (C = 192) against fp64 autograd: the GEMM-composed backward (AUTO) and the SIMT
    kernel, NCHW and channels-last, 32,768 and 1,961 pixels per image"""
    p, gy, ref = _gdn_reference(GDN_SHAPES[shape], inverse)
    got, path = _gdn_backward(pkg, lib, cuda_dev, p, gy, inverse, algo, channels_last)
    assert path == ("composed" if algo == ALGO_AUTO else "simt")
    _check_gdn(got, ref, record_property)


@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
@pytest.mark.parametrize("inverse", [False, True], ids=["gdn", "igdn"])
@pytest.mark.parametrize("shape", list(GDN_SHAPES))
def test_gdn_backward_auto_matches_simt(cuda_dev, pkg, lib, record_property, shape, inverse, channels_last):
    """the two backward implementations agree to 1e-5 of each gradient's largest magnitude"""
    p, gy, _ = _gdn_reference(GDN_SHAPES[shape], inverse)
    auto, _ = _gdn_backward(pkg, lib, cuda_dev, p, gy, inverse, ALGO_AUTO, channels_last)
    simt, _ = _gdn_backward(pkg, lib, cuda_dev, p, gy, inverse, ALGO_SIMT, channels_last)
    for k in ("x", "beta", "gamma"):
        r = _max_rel(auto[k], simt[k])
        record_property(f"auto_vs_simt_{k}", r)
        assert r <= 1e-5, f"d{k}: AUTO and SIMT differ by {r:.3e} relative"


@pytest.mark.parametrize("channels_last", [False, True], ids=["nchw", "nhwc"])
def test_gdn_backward_lower_bound_rule(cuda_dev, pkg, lib, record_property, channels_last):
    """C = 16 with beta / gamma entries below their bounds (and one negative gamma) on the composed path: the LowerBound
    pass-through rule of gdn_bwd_finalize (gradient kept where the parameter is at or above the bound or the gradient
    is negative)"""
    p, gy, ref = _gdn_reference((2, 16, 40, 56), False, hit_bounds=True)
    got, path = _gdn_backward(pkg, lib, cuda_dev, p, gy, False, ALGO_AUTO, channels_last)
    assert path == "composed"
    clamped_b = p["beta"] < 1e-3
    assert bool(clamped_b.any()) and bool((ref["beta"][clamped_b] == 0).any())       # the rule zeroes some of them
    _check_gdn(got, ref, record_property)


def test_gdn_backward_odd_numel_falls_back_to_simt(cuda_dev, pkg, lib, record_property):
    """numel % 4 != 0 (the composed stages are float4-vectorised): AUTO runs the SIMT kernel"""
    p, gy, ref = _gdn_reference((1, 5, 3, 3), False)
    got, path = _gdn_backward(pkg, lib, cuda_dev, p, gy, False, ALGO_AUTO, False)
    assert path == "simt"
    _check_gdn(got, ref, record_property)
