"""CPU restatement of the reference hot path (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py).

Written from the semantics in SURVEY.md Appendix A, one function per row of section 8(a); every
function cites the reference lines it restates.  It is deliberately *not* structured like the
reference code: windows are addressed by coordinates, the keep predicate and the SW-MSA mask
are computed per window from (row, col) bands, and nothing is gathered / scattered through
boolean indexing.  Pinned by tests/golden (outputs of the reference itself) and by
tests/test_oracle_vs_reference.py when /root/reference is importable.

All functions take/return torch CPU tensors and compute in the dtype of their inputs
(fp32 = what the reference computes; fp64 = tight yardstick for the tolerance tests).
"""
from __future__ import annotations

import math

import torch

NEG_MASK = -100.0  # layers/masked_win_attention.py:214


# --------------------------------------------------------------------------------------
# a4: window partition / reverse   (layers/masked_win_attention.py:6-33)
# --------------------------------------------------------------------------------------
def to_windows(x_nhwc: torch.Tensor, ws: int) -> torch.Tensor:
    """(B,H,W,C) -> (B*nWh*nWw, ws, ws, C); window order (b, wh, ww) row-major."""
    B, H, W, C = x_nhwc.shape
    if H % ws or W % ws:
        raise RuntimeError(f"H={H}, W={W} must be multiples of window_size={ws}")
    t = x_nhwc.reshape(B, H // ws, ws, W // ws, ws, C)
    return t.permute(0, 1, 3, 2, 4, 5).reshape(-1, ws, ws, C)


def from_windows(win: torch.Tensor, ws: int, H: int, W: int) -> torch.Tensor:
    """inverse of to_windows: (B*nW, ws, ws, C) -> (B,H,W,C)."""
    nh, nw = H // ws, W // ws
    B = win.shape[0] // (nh * nw)
    t = win.reshape(B, nh, nw, ws, ws, -1)
    return t.permute(0, 1, 3, 2, 4, 5).reshape(B, H, W, -1)


# --------------------------------------------------------------------------------------
# relative position index / bias   (layers/masked_win_attention.py:72-86, 109-112)
# --------------------------------------------------------------------------------------
def relative_position_index(ws: int) -> torch.Tensor:
    """idx[i,j] = (yi-yj+ws-1)*(2ws-1) + (xi-xj+ws-1), tokens row-major in the window."""
    t = torch.arange(ws * ws)
    ty, tx = t // ws, t % ws
    dy = ty[:, None] - ty[None, :] + ws - 1
    dx = tx[:, None] - tx[None, :] + ws - 1
    return dy * (2 * ws - 1) + dx


def expand_bias(table: torch.Tensor, ws: int) -> torch.Tensor:
    """((2ws-1)^2, h) parameter -> (h, N, N) additive bias."""
    N = ws * ws
    idx = relative_position_index(ws).reshape(-1)
    return table[idx].reshape(N, N, -1).permute(2, 0, 1).contiguous()


# --------------------------------------------------------------------------------------
# a5: SW-MSA region mask   (layers/masked_win_attention.py:194-216, win_attention.py:159-179)
# --------------------------------------------------------------------------------------
def _band(coord: torch.Tensor, size: int, ws: int, s: int) -> torch.Tensor:
    # slices (0,-ws) | (-ws,-s) | (-s,None) in the SHIFTED frame
    return (coord >= size - ws).long() + (coord >= size - s).long()


def shift_region_mask(H: int, W: int, ws: int, s: int, dtype=torch.float32) -> torch.Tensor:
    """(nWh*nWw, N, N): 0 where the two tokens share a region id, -100 otherwise."""
    ys = torch.arange(H)
    xs = torch.arange(W)
    rid = 3 * _band(ys, H, ws, s)[:, None] + _band(xs, W, ws, s)[None, :]      # (H, W)
    rid = to_windows(rid.reshape(1, H, W, 1), ws).reshape(-1, ws * ws)          # (nW, N)
    differ = rid[:, :, None] != rid[:, None, :]
    return differ.to(dtype) * NEG_MASK


# --------------------------------------------------------------------------------------
# a3: keep predicate   (layers/masked_win_attention.py:35-47)
# --------------------------------------------------------------------------------------
def window_keep(alpha: torch.Tensor, ws: int, s: int) -> torch.Tensor:
    """alpha (B,1,H,W) -> bool (B*nW,): window kept iff its (cyclically shifted) alpha sums != 0."""
    a = alpha.permute(0, 2, 3, 1)
    if s > 0:
        a = torch.roll(a, shifts=(-s, -s), dims=(1, 2))
    return to_windows(a, ws).sum(dim=(1, 2, 3)) != 0


# --------------------------------------------------------------------------------------
# a2: window attention core   (layers/masked_win_attention.py:96-131)
# --------------------------------------------------------------------------------------
def window_attention(xw, qkv_w, qkv_b, proj_w, proj_b, bias_table, heads: int, ws: int,
                     mask=None, qk_scale=None):
    """xw (K,N,C) -> (K,N,C).  mask: None or (K,N,N) additive (already per kept window)."""
    K, N, C = xw.shape
    d = C // heads
    scale = qk_scale or d ** -0.5
    qkv = xw @ qkv_w.t()
    if qkv_b is not None:
        qkv = qkv + qkv_b
    qkv = qkv.reshape(K, N, 3, heads, d)
    q = qkv[:, :, 0].permute(0, 2, 1, 3) * scale      # (K,h,N,d); the reference scales q after the projection
    k = qkv[:, :, 1].permute(0, 2, 1, 3)
    v = qkv[:, :, 2].permute(0, 2, 1, 3)
    s_ = torch.einsum("khid,khjd->khij", q, k)
    s_ = s_ + expand_bias(bias_table, ws).to(s_.dtype)[None]
    if mask is not None:
        s_ = s_ + mask[:, None]
    p = torch.softmax(s_, dim=-1)
    o = torch.einsum("khij,khjd->kihd", p, v).reshape(K, N, C)
    return o @ proj_w.t() + proj_b


# --------------------------------------------------------------------------------------
# a1 / a6: the full block   (layers/masked_win_attention.py:169-251, win_attention.py:153-207)
# --------------------------------------------------------------------------------------
def masked_window_attention(x, alpha, qkv_w, qkv_b, proj_w, proj_b, bias_table,
                            heads: int, ws: int, shift: int, qk_scale=None):
    """x (B,C,H,W), alpha (B,1,H,W) or None (= unmasked twin, every window kept) -> (B,C,H,W)."""
    assert 0 <= shift < ws, "shift_size must in 0-window_size"
    B, C, H, W = x.shape
    xs = x.permute(0, 2, 3, 1)
    if shift > 0:
        xs = torch.roll(xs, shifts=(-shift, -shift), dims=(1, 2))
    xw = to_windows(xs, ws).reshape(-1, ws * ws, C)                              # (B*nW, N, C)
    nW = (H // ws) * (W // ws)
    if alpha is None:
        keep = torch.ones(B * nW, dtype=torch.bool)
    else:
        keep = window_keep(alpha, ws, shift)
    mask = None
    if shift > 0:
        mask = shift_region_mask(H, W, ws, shift, x.dtype).repeat(B, 1, 1)[keep]
    y = torch.zeros_like(xw)
    if bool(keep.any()):
        y[keep] = window_attention(xw[keep], qkv_w, qkv_b, proj_w, proj_b, bias_table,
                                   heads, ws, mask=mask, qk_scale=qk_scale)
    ys = from_windows(y.reshape(-1, ws, ws, C), ws, H, W)
    if shift > 0:
        ys = torch.roll(ys, shifts=(shift, shift), dims=(1, 2))
    return x + ys.permute(0, 3, 1, 2)


# --------------------------------------------------------------------------------------
# a8: LowerBound   (layers/GDN.py:9-23)
# --------------------------------------------------------------------------------------
class _LowerBound(torch.autograd.Function):
    @staticmethod
    def forward(ctx, v, bound):
        ctx.save_for_backward(v)
        ctx.bound = bound
        return torch.clamp_min(v, bound)

    @staticmethod
    def backward(ctx, g):
        (v,) = ctx.saved_tensors
        # fp32 comparison against fp32(bound), as `ones_like(inputs) * bound` does
        b = torch.full_like(v, ctx.bound)
        return torch.where((v >= b) | (g < 0), g, torch.zeros_like(g)), None


def lower_bound(v, bound: float):
    return _LowerBound.apply(v, bound)


# --------------------------------------------------------------------------------------
# a7: GDN / IGDN   (layers/GDN.py:46-94)
# --------------------------------------------------------------------------------------
def gdn_constants(beta_min=1e-6, reparam_offset=2 ** -18):
    pedestal = reparam_offset ** 2
    return pedestal, (beta_min + pedestal) ** 0.5, reparam_offset   # pedestal, beta_bound, gamma_bound


def gdn_effective_params(beta_p, gamma_p, beta_min=1e-6, reparam_offset=2 ** -18):
    pedestal, beta_bound, gamma_bound = gdn_constants(beta_min, reparam_offset)
    beta = lower_bound(beta_p, beta_bound) ** 2 - pedestal
    gamma = lower_bound(gamma_p, gamma_bound) ** 2 - pedestal
    return beta, gamma


def gdn(x, beta_p, gamma_p, inverse=False, beta_min=1e-6, reparam_offset=2 ** -18):
    """x (B,C,H,W) [or (B,C,D,W,H)] ; n_i = beta_i + sum_j gamma[i,j] x_j^2 ; y = x * n^(-/+ 1/2)."""
    shape = x.shape
    if x.dim() == 5:
        x = x.reshape(shape[0], shape[1], shape[2] * shape[3], shape[4])
    beta, gamma = gdn_effective_params(beta_p, gamma_p, beta_min, reparam_offset)
    n = torch.einsum("ij,bjhw->bihw", gamma, x * x) + beta[None, :, None, None]
    r = torch.sqrt(n)
    y = x * r if inverse else x / r
    return y.reshape(shape)


# --------------------------------------------------------------------------------------
# a9: latent rounding   (models/AutoEncoderRGB_Journal.py:31-32, 212-214, 227-229, 257, 263-264)
# --------------------------------------------------------------------------------------
def ste_round(x):
    """forward value of `round(x) - x.detach() + x` (round-half-even), identity gradient."""
    return torch.round(x) - x.detach() + x


def quantize_offset(x, mu):
    """z_hat = ste_round(z - med) + med ; y_hat = ste_round(y - mu) + mu."""
    return ste_round(x - mu) + mu


def lrp_add(y_hat, lrp):
    """y_hat + 0.5 * tanh(lrp)   (models/AutoEncoderRGB_Journal.py:262-264)."""
    return y_hat + 0.5 * torch.tanh(lrp)


def quantize_levels(m, levels: int = 255):
    """reconmask = round(m * 255) / 255   (models/AutoEncoderRGB_Journal.py:212-214)."""
    return torch.round(m * levels) / levels


# --------------------------------------------------------------------------------------
# alpha pyramid feeding a1   (layers/SupplyMask.py:7-18) -- input generator for the benches
# --------------------------------------------------------------------------------------
def gate_residual(a, b, x):
    """layers/Masked_Attention.py:186-188:  out = a * torch.sigmoid(b); out += identity."""
    return a * torch.sigmoid(b) + x


def _residual_unit(x, w, prefix):
    """layers/Masked_Attention.py:150-171: conv1x1 -> GELU -> conv3x3 -> GELU -> conv1x1, + identity, GELU."""
    F = torch.nn.functional
    out = F.conv2d(x, w[prefix + "conv.0.weight"], w[prefix + "conv.0.bias"])
    out = F.gelu(out)
    out = F.conv2d(out, w[prefix + "conv.2.weight"], w[prefix + "conv.2.bias"], padding=1)
    out = F.gelu(out)
    out = F.conv2d(out, w[prefix + "conv.4.weight"], w[prefix + "conv.4.bias"])
    return F.gelu(out + x)


def win_noshift_attention(x, mask, w, heads: int, ws: int, shift: int):
    """layers/Masked_Attention.py:182-189 (Win_noShift_Attention.forward) on a reference-style state dict `w`."""
    a = x
    for i in range(3):
        a = _residual_unit(a, w, f"conv_a.{i}.")
    b = masked_window_attention(x, mask, w["attn.attn.qkv.weight"], w.get("attn.attn.qkv.bias"),
                                w["attn.attn.proj.weight"], w["attn.attn.proj.bias"],
                                w["attn.attn.relative_position_bias_table"], heads, ws, shift)
    for i in range(3):
        b = _residual_unit(b, w, f"conv_b.{i}.")
    b = torch.nn.functional.conv2d(b, w["conv_b.3.weight"], w["conv_b.3.bias"])
    return gate_residual(a, b, x)


def alpha_pyramid(alpha, levels: int = 6):
    out = []
    a = alpha
    for _ in range(levels):
        a = torch.nn.functional.avg_pool2d(a, 3, stride=2, padding=1)   # count_include_pad=True
        out.append(a)
    return out


def constraint(t):
    """isolated-pixel clean-up of the decoded mask (trainRGB.py:98-111 = trainmask.py:133-146): both masks are taken from
    the tensor before either assignment; returns a new tensor"""
    kernel = torch.ones(1, 1, 3, 3, dtype=t.dtype)
    kernel[0, 0, 1, 1] = 0
    B, C, H, W = t.shape
    nsum = torch.nn.functional.conv2d(t.reshape(B * C, 1, H, W), kernel, padding=1).reshape(B, C, H, W)
    out = t.clone()
    out[(t == 0) & (nsum == 8)] = 1
    out[(t > 0) & (nsum == 0)] = 0
    return out


def flops_per_window(C: int, ws: int) -> int:
    N = ws * ws
    return 8 * N * C * C + 4 * N * N * C


__all__ = [n for n in dir() if not n.startswith("_") and n not in ("annotations", "math", "torch")]
