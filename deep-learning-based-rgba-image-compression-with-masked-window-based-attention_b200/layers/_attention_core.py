"""Shared machinery of the two window-attention drop-ins (masked / unmasked).

Forward = the fused sm_100a kernel (`mwa_forward`, `window_attention_forward`).
Backward (training, BASELINE config 5) = the hand-written `mwa_backward` / `window_attention_backward`
kernels (fp32; they re-compute q, k, v and the softmax per head, emit grad_x and the relative-position
table gradient, and leave four token-major scratch tensors), followed by the weight / bias gradients
as plain GEMMs and column sums over all tokens (library GEMM: `dWqkv = dqkv^T xw`, `dWproj = dy^T ao`).
With `algo = ALGO_SIMT` one all-in-one kernel does the token GEMMs too; otherwise (default) the three token GEMMs
(qkv recompute, dAO = dy Wproj, dXw = dqkv Wqkv) run in the library GEMM as well and hand-written gather / per-window
core / scatter kernels do the rest (3.5x faster).
"""
from __future__ import annotations

import torch
from torch import nn
from torch.autograd import Function

from .. import _abi
from ._params import ParamBlock, ParamBlockOwner
from .conv import gemm_tokens


def _window_partition(x, window_size):
    B, H, W, C = x.shape
    x = x.view(B, H // window_size, window_size, W // window_size, window_size, C)
    return x.permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, window_size, window_size, C)


def _window_reverse(windows, window_size, H, W):
    B = int(windows.shape[0] / (H * W / window_size / window_size))
    x = windows.view(B, H // window_size, W // window_size, window_size, window_size, -1)
    return x.permute(0, 1, 3, 2, 4, 5).contiguous().view(B, H, W, -1)


class WindowAttentionFunction(Function):
    """out = x + window_attention(x) on kept windows; alpha=None keeps every window."""

    @staticmethod
    def forward(ctx, x, alpha, qkv_w, qkv_b, proj_w, proj_b, table, attn_mod, ws, shift, algo):
        lib = _abi.load()
        _abi.require_cuda_f32(x, "attention input")
        if alpha is not None:
            _abi.require_cuda_f32(alpha, "img_alpha")
        B, C, H, W = x.shape
        if H % ws or W % ws:
            # the reference fails in window_partition's .view (layers/masked_win_attention.py:15)
            raise RuntimeError(f"shape '[{B}, {H // ws}, {ws}, {W // ws}, {ws}, {C}]' is invalid for input of size "
                               f"{x.numel()}: H={H}, W={W} must be multiples of window_size={ws}")
        if x.numel() == 0:                   # empty batch: nothing to launch (data_ptr() of an empty tensor is null)
            ctx.empty = True
            return torch.empty_like(x)
        ctx.empty = False
        channels_last = (not x.is_contiguous()) and x.is_contiguous(memory_format=torch.channels_last)
        # The fp32-faithful fast kernels read NCHW.  A channels-last input goes through them too (one transposing copy
        # each way: far cheaper than the general SIMT kernel, which is what the C ABI falls back to for NHWC); the output
        # keeps the input's memory format, as torch ops do.  Only the general SIMT kernel consumes NHWC in place.
        relayout = channels_last and algo in (_abi.ALGO_AUTO, _abi.ALGO_TCGEN05) and \
            bool(lib.mwa_fast_path_needs_nchw(C, attn_mod.num_heads, ws))
        if relayout or not channels_last:
            x = x.contiguous()
            channels_last = False
        if alpha is not None:
            if alpha.shape != (B, 1, H, W):
                raise RuntimeError(f"img_alpha must have shape {(B, 1, H, W)}, got {tuple(alpha.shape)}")
            alpha = alpha.contiguous()       # (B,1,H,W): NCHW and NHWC coincide
        with torch.cuda.device(x.device):
            blk = attn_mod._param_block(qkv_w, qkv_b, proj_w, proj_b, table)
            out = torch.empty_like(x)
            wsp = torch.empty(int(lib.mwa_workspace_bytes(B, H, W, ws)), dtype=torch.uint8, device=x.device)
            _abi.check(lib.mwa_forward(x.data_ptr(), _abi.ptr(alpha), out.data_ptr(), blk.data_ptr(), B, C, H, W,
                                       attn_mod.num_heads, ws, shift, int(channels_last), algo, None,
                                       wsp.data_ptr(), wsp.numel(), _abi.stream_handle()), "mwa_forward")
        if relayout:
            out = out.contiguous(memory_format=torch.channels_last)
        ctx.cfg = (attn_mod, ws, shift)
        ctx.algo = algo
        ctx.has_bias = qkv_b is not None
        ctx.save_for_backward(x, alpha, qkv_w, qkv_b, proj_w, proj_b, table)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        if ctx.empty:
            return (grad_out,) + (None,) * 10
        x, alpha, qkv_w, qkv_b, proj_w, proj_b, table = ctx.saved_tensors
        attn_mod, ws, shift = ctx.cfg
        lib = _abi.load()
        _abi.require_cuda_f32(grad_out, "grad_output")
        B, C, H, W = x.shape
        channels_last = (not x.is_contiguous()) and x.is_contiguous(memory_format=torch.channels_last)
        grad_out = grad_out.contiguous(memory_format=torch.channels_last) if channels_last else grad_out.contiguous()
        N, nwin = ws * ws, B * (H // ws) * (W // ws)
        with torch.cuda.device(x.device):
            blk = attn_mod._param_block(qkv_w, qkv_b, proj_w, proj_b, table)
            gx = torch.empty_like(x)
            gtab = torch.empty_like(table)
            xw, ao, dy = (torch.empty(nwin * N, C, device=x.device) for _ in range(3))
            dqkv = torch.empty(nwin * N, 3 * C, device=x.device)
            qw, pw = qkv_w.contiguous(), proj_w.contiguous()
            st = _abi.stream_handle()
            if ctx.algo == _abi.ALGO_SIMT:
                # everything in one hand-written kernel (token GEMMs included)
                _abi.check(lib.mwa_backward(x.data_ptr(), _abi.ptr(alpha), grad_out.data_ptr(), qw.data_ptr(),
                                            pw.data_ptr(), blk.data_ptr(), gx.data_ptr(), gtab.data_ptr(),
                                            xw.data_ptr(), ao.data_ptr(), dy.data_ptr(), dqkv.data_ptr(), B, C, H, W,
                                            attn_mod.num_heads, ws, shift, int(channels_last), st), "mwa_backward")
            else:
                # gather -> token GEMMs (library) -> per-window core kernel -> token GEMM -> scatter
                flags = torch.empty(max(nwin, 1), dtype=torch.uint8, device=x.device)
                _abi.check(lib.mwa_bwd_gather(x.data_ptr(), _abi.ptr(alpha), grad_out.data_ptr(), xw.data_ptr(),
                                              dy.data_ptr(), flags.data_ptr(), B, C, H, W, ws, shift,
                                              int(channels_last), st), "mwa_bwd_gather")
                # the token GEMMs on the convolution kernel (fp32-faithful tcgen05; gradients pre-scaled by a power of two)
                qkv = gemm_tokens(xw, qw, qkv_b)
                dao = gemm_tokens(dy, pw, weight_is_in_out=True, scale_input=True)
                _abi.check(lib.mwa_bwd_core(qkv.data_ptr(), dao.data_ptr(), blk.data_ptr(), None, flags.data_ptr(),
                                            ao.data_ptr(), dqkv.data_ptr(), gtab.data_ptr(), nwin, C, H, W,
                                            attn_mod.num_heads, ws, shift, 0, st), "mwa_bwd_core")
                dxw = gemm_tokens(dqkv, qw, weight_is_in_out=True, scale_input=True)
                _abi.check(lib.mwa_bwd_scatter(grad_out.data_ptr(), dxw.data_ptr(), gx.data_ptr(), B, C, H, W, ws,
                                               shift, int(channels_last), st), "mwa_bwd_scatter")
            need = ctx.needs_input_grad
            with _abi.tf32_reduction(nwin * N):          # K = all tokens
                gw1 = dqkv.t() @ xw if need[2] else None
                gw2 = dy.t() @ ao if need[4] else None
            gb1 = dqkv.sum(0) if (need[3] and ctx.has_bias) else None
            gb2 = dy.sum(0) if need[5] else None
        return (gx if need[0] else None), None, gw1, gb1, gw2, gb2, (gtab if need[6] else None), None, None, None, None


class TokenAttentionFunction(Function):
    """WindowAttention.forward on (K, N, C) tokens with an optional additive (nW, N, N) mask (no residual)."""

    @staticmethod
    def forward(ctx, xw, mask, qkv_w, qkv_b, proj_w, proj_b, table, attn_mod):
        lib = _abi.load()
        _abi.require_cuda_f32(xw, "window tokens")
        K, N, C = xw.shape
        ws = attn_mod.window_size[0]
        if attn_mod.window_size[0] != attn_mod.window_size[1] or N != ws * ws:
            raise RuntimeError(f"expected {ws * ws} tokens per window, got {N}")
        xw = xw.contiguous()
        nw = 0
        if mask is not None:
            _abi.require_cuda_f32(mask, "mask")
            mask = mask.contiguous()
            nw = mask.shape[0]
            if nw == 0:
                print("nW error!")           # layers/masked_win_attention.py:116-118
                mask, nw = None, 0
            elif K % nw != 0 or mask.shape[1:] != (N, N):
                raise RuntimeError(f"mask of shape {tuple(mask.shape)} does not tile {K} windows")
        with torch.cuda.device(xw.device):
            blk = attn_mod._param_block(qkv_w, qkv_b, proj_w, proj_b, table)
            out = torch.empty_like(xw)
            _abi.check(lib.window_attention_forward(xw.data_ptr(), _abi.ptr(mask), out.data_ptr(), blk.data_ptr(), K, C,
                                                    attn_mod.num_heads, ws, nw, _abi.stream_handle()),
                       "window_attention_forward")
        ctx.attn_mod = attn_mod
        ctx.save_for_backward(xw, mask, qkv_w, qkv_b, proj_w, proj_b, table)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        xw, mask, qkv_w, qkv_b, proj_w, proj_b, table = ctx.saved_tensors
        m = ctx.attn_mod
        lib = _abi.load()
        _abi.require_cuda_f32(grad_out, "grad_output")
        grad_out = grad_out.contiguous()
        K, N, C = xw.shape
        ws = m.window_size[0]
        nw = 0 if mask is None else mask.shape[0]
        with torch.cuda.device(xw.device):
            blk = m._param_block(qkv_w, qkv_b, proj_w, proj_b, table)
            gx = torch.empty_like(xw)
            gtab = torch.empty_like(table)
            ao = torch.empty(K * N, C, device=xw.device)
            dqkv = torch.empty(K * N, 3 * C, device=xw.device)
            qw, pw = qkv_w.contiguous(), proj_w.contiguous()
            xf, dyf = xw.reshape(K * N, C), grad_out.reshape(K * N, C)
            if getattr(m, "algo", _abi.ALGO_AUTO) == _abi.ALGO_SIMT:
                _abi.check(lib.window_attention_backward(xw.data_ptr(), _abi.ptr(mask), grad_out.data_ptr(),
                                                         qw.data_ptr(), pw.data_ptr(), blk.data_ptr(), gx.data_ptr(),
                                                         gtab.data_ptr(), ao.data_ptr(), dqkv.data_ptr(), K, C,
                                                         m.num_heads, ws, nw, _abi.stream_handle()),
                           "window_attention_backward")
            else:
                qkv = gemm_tokens(xf.contiguous(), qw, qkv_b)
                dao = gemm_tokens(dyf.contiguous(), pw, weight_is_in_out=True, scale_input=True)
                _abi.check(lib.mwa_bwd_core(qkv.data_ptr(), dao.data_ptr(), blk.data_ptr(), _abi.ptr(mask), None,
                                            ao.data_ptr(), dqkv.data_ptr(), gtab.data_ptr(), K, C, 0, 0, m.num_heads,
                                            ws, 0, nw, _abi.stream_handle()), "mwa_bwd_core")
                gx = gemm_tokens(dqkv, qw, weight_is_in_out=True, scale_input=True).view(K, N, C)
            need = ctx.needs_input_grad
            with _abi.tf32_reduction(K * N):
                gw1 = dqkv.t() @ xf if need[2] else None
                gw2 = dyf.t() @ ao if need[4] else None
            gb1 = dqkv.sum(0) if (need[3] and qkv_b is not None) else None
            gb2 = dyf.sum(0) if need[5] else None
        return (gx if need[0] else None), None, gw1, gb1, gw2, gb2, (gtab if need[6] else None), None


class WindowAttentionBase(ParamBlockOwner, nn.Module):
    """Window based multi-head self attention (W-MSA) with relative position bias -- parameter container and
    token-level forward.  Same constructor / attributes / state-dict keys as the reference class
    (layers/masked_win_attention.py:49-131 == layers/win_attention.py:37-115)."""

    def __init__(self, dim=192, window_size=(8, 8), num_heads=8, qkv_bias=True, qk_scale=None, attn_drop=0.,
                 proj_drop=0.):
        super().__init__()
        if attn_drop != 0. or proj_drop != 0.:
            raise NotImplementedError("the fused sm_100a kernel implements attn_drop = proj_drop = 0 "
                                      "(the only values the reference models use)")
        if dim % num_heads != 0:
            raise ValueError(f"dim={dim} must be divisible by num_heads={num_heads}")
        self.dim = dim
        self.window_size = tuple(window_size)
        self.num_heads = num_heads
        head_dim = dim // num_heads
        self.scale = qk_scale or head_dim ** -0.5

        self.relative_position_bias_table = nn.Parameter(
            torch.zeros((2 * window_size[0] - 1) * (2 * window_size[1] - 1), num_heads))

        t = torch.arange(window_size[0] * window_size[1])
        ty, tx = t // window_size[1], t % window_size[1]
        rel = (ty[:, None] - ty[None, :] + window_size[0] - 1) * (2 * window_size[1] - 1) \
            + (tx[:, None] - tx[None, :] + window_size[1] - 1)
        self.register_buffer("relative_position_index", rel)

        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.attn_drop = nn.Dropout(attn_drop)
        self.proj = nn.Linear(dim, dim)
        self.proj_drop = nn.Dropout(proj_drop)
        nn.init.trunc_normal_(self.relative_position_bias_table, std=.02)
        self.softmax = nn.Softmax(dim=-1)
        self._blk = ParamBlock()

    def _param_block(self, qkv_w, qkv_b, proj_w, proj_b, table):
        lib = _abi.load()
        if self.window_size[0] != self.window_size[1]:
            raise NotImplementedError("square windows only (the reference only builds square windows)")
        C, h, ws = self.dim, self.num_heads, self.window_size[0]
        for name, t in (("qkv.weight", qkv_w), ("proj.weight", proj_w), ("proj.bias", proj_b),
                        ("relative_position_bias_table", table)):
            _abi.require_cuda_f32(t, name)
        nbytes = int(lib.mwa_param_bytes(C, h, ws))

        def fill(blk):
            _abi.check(lib.mwa_prepare(qkv_w.data_ptr(), _abi.ptr(qkv_b), proj_w.data_ptr(), proj_b.data_ptr(),
                                       table.data_ptr(), C, h, ws, float(self.scale), blk.data_ptr(), blk.numel(),
                                       _abi.stream_handle()), "mwa_prepare")

        return self._blk.get((qkv_w, qkv_b, proj_w, proj_b, table), nbytes, fill)

    def forward(self, x, mask=None):
        """x: (num_windows*B, N, C); mask: (num_windows, N, N) additive or None."""
        self._refresh_if_training()
        return TokenAttentionFunction.apply(x, mask, self.qkv.weight, self.qkv.bias, self.proj.weight,
                                            self.proj.bias, self.relative_position_bias_table, self)
