"""Evaluation metrics of the RGBA codec on the B200 (SURVEY.md section 8f, rank 4).

    masked_ms_ssim(X, Y, mask, data_range=1.0)   metrics/masked_ms_ssim_torch.py:181-265  ms_ssim(X, Y, mask, data_range)
    masked_psnr(X, Y, mask)                      models/AutoEncoderRGB_Journal.py:36-64 + trainRGB.py:303

Two kernel launches per MS-SSIM level (csrc/msssim.cu) instead of the reference's ~40 torch kernels; no host
synchronisation: the result is a 0-dim tensor on the device.  When X or Y requires grad, the metric is differentiable in
both (one backward launch per level, no host synchronisation either), so it can be a training loss.
"""
from __future__ import annotations

import torch
from torch.autograd.function import once_differentiable

from . import _abi

MS_SSIM_WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)


def _levels(X, Y, m, data_range, n):
    """the metric's launches, level by level: yields (per, X_l, Y_l, m_l, cnt) with per (B, C, 2) = (S, CS) of level l;
    the pool that feeds level l + 1 is launched when the next level is asked for"""
    lib = _abi.load()
    B, C, H, W = X.shape
    st = _abi.stream_handle()
    with torch.cuda.device(X.device):
        for lvl in range(n):
            sums = torch.empty(B, C, 2, device=X.device, dtype=torch.float32)
            cnt = torch.empty(B, device=X.device, dtype=torch.float32)
            _abi.check(lib.ms_ssim_level_forward(X.data_ptr(), Y.data_ptr(), m.data_ptr(), B, C, H, W, float(data_range),
                                                 sums.data_ptr(), cnt.data_ptr(), st), "ms_ssim_level_forward")
            yield sums / (cnt.view(B, 1, 1) + 1e-10), X, Y, m, cnt
            if lvl < n - 1:
                Hp, Wp = (H + 2 * (H % 2) - 2) // 2 + 1, (W + 2 * (W % 2) - 2) // 2 + 1
                Xo = torch.empty(B, C, Hp, Wp, device=X.device, dtype=torch.float32)
                Yo, Mo = torch.empty_like(Xo), torch.empty(B, Hp, Wp, device=X.device, dtype=torch.float32)
                _abi.check(lib.ms_ssim_pool_forward(X.data_ptr(), Y.data_ptr(), m.data_ptr(), B, C, H, W, Xo.data_ptr(),
                                                    Yo.data_ptr(), Mo.data_ptr(), st), "ms_ssim_pool_forward")
                X, Y, m, H, W = Xo, Yo, Mo, Hp, Wp


class _MsSsimLevels(torch.autograd.Function):
    """(X, Y, mask) -> (n, B, C, 2): the per-level (S, CS) of the masked MS-SSIM.  The forward is the metric's launches;
    the backward is one ms_ssim_level_backward launch per level, coarsest first, each adding the adjoint of the pool to
    the next level.  It recomputes the levels' maps from the saved level inputs and makes no host synchronisation."""

    @staticmethod
    def forward(ctx, X, Y, m, data_range, n):
        pers, saved = [], []
        for per, *level in _levels(X, Y, m, data_range, n):
            pers.append(per)
            saved += level
        ctx.save_for_backward(*saved)
        ctx.data_range = data_range
        return torch.stack(pers)

    @staticmethod
    @once_differentiable
    def backward(ctx, grad):
        lib = _abi.load()
        grad = grad.contiguous()
        saved = ctx.saved_tensors
        want_x, want_y = ctx.needs_input_grad[:2]
        dXc = dYc = None
        st = _abi.stream_handle()
        with torch.cuda.device(grad.device):
            for lvl in reversed(range(grad.shape[0])):
                X, Y, m, cnt = saved[4 * lvl:4 * lvl + 4]
                B, C, H, W = X.shape
                dX = torch.empty_like(X) if want_x else None
                dY = torch.empty_like(Y) if want_y else None
                _abi.check(lib.ms_ssim_level_backward(X.data_ptr(), Y.data_ptr(), m.data_ptr(), B, C, H, W, ctx.data_range,
                                                      grad[lvl].data_ptr(), cnt.data_ptr(), _abi.ptr(dXc), _abi.ptr(dYc),
                                                      _abi.ptr(dX), _abi.ptr(dY), st), "ms_ssim_level_backward")
                dXc, dYc = dX, dY
        return dXc, dYc, None, None, None


def masked_ms_ssim(X: torch.Tensor, Y: torch.Tensor, mask: torch.Tensor, data_range: float = 1.0,
                   weights=MS_SSIM_WEIGHTS) -> torch.Tensor:
    """Differentiable in X and Y (not in the mask): `1 - masked_ms_ssim(x_hat, image, mask)` is a distortion term."""
    for name, t in (("X", X), ("Y", Y), ("mask", mask)):
        _abi.require_cuda_f32(t, f"masked_ms_ssim {name}")
    if X.shape != Y.shape or X.dim() != 4:
        raise RuntimeError(f"masked_ms_ssim: X {tuple(X.shape)} and Y {tuple(Y.shape)} must be equal (B, C, H, W)")
    B, C, H, W = X.shape
    if mask.numel() != B * H * W:
        raise RuntimeError(f"masked_ms_ssim: mask {tuple(mask.shape)} must be (B, 1, H, W)")
    if min(H, W) <= (11 - 1) * 2 ** 4:
        # the reference's assertion (metrics/masked_ms_ssim_torch.py:222-225)
        raise AssertionError("Image size should be larger than 160 due to the 4 downsamplings in ms-ssim")
    X, Y, m = X.contiguous(), Y.contiguous(), mask.reshape(B, H, W).contiguous()
    n = len(weights)
    if torch.is_grad_enabled() and (X.requires_grad or Y.requires_grad):
        per = _MsSsimLevels.apply(X, Y, m.detach(), float(data_range), n)
        # the weighted product as n - 1 multiplications with scalar exponents: the same function and the same gradient at
        # relu(0) as prod(stack ** w), but torch.prod's backward reads its zero count on the host (one sync per step)
        out = None
        for lvl, wt in enumerate(weights):
            v = torch.relu(per[lvl, ..., 1] if lvl < n - 1 else per[lvl, ..., 0]) ** wt
            out = v if out is None else out * v
        return out.mean()
    vals = []
    for lvl, (per, *_) in enumerate(_levels(X, Y, m, data_range, n)):
        vals.append(torch.relu(per[..., 1] if lvl < n - 1 else per[..., 0]))
    w = torch.tensor(weights, device=X.device, dtype=torch.float32).view(-1, 1, 1)
    return torch.prod(torch.stack(vals, 0) ** w, dim=0).mean()


def masked_mse(X: torch.Tensor, Y: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """squared error over the pixels whose alpha is > 0, per image, averaged (models/AutoEncoderRGB_Journal.py:36-64)"""
    m = (mask.expand(-1, X.shape[1], -1, -1) > 0).to(X.dtype)
    se = ((X * m - Y * m) ** 2).sum(dim=(1, 2, 3))
    return torch.mean(se / torch.clamp(m.sum(dim=(1, 2, 3)), min=1))


def masked_psnr(X: torch.Tensor, Y: torch.Tensor, mask: torch.Tensor) -> torch.Tensor:
    """trainRGB.py:303"""
    return 10.0 * torch.log10(1.0 / masked_mse(X, Y, mask))
