"""The callers of the hot path, assembled on the B200 modules: the RGBA codec's encode + decode forward.

The reference's own model files (models/AutoEncoderRGB_Journal.py, layers/TransformRGB.py) build on the drop-in modules
unchanged once `install()` has re-bound `layers.*` -- that is the integration route when the reference tree is present
(INTEGRATION.md).  This file is the same module tree written against the drop-ins directly, for boxes where the reference
is absent (the GPU box of the test / bench harness): identical attribute names and state-dict keys
(`Encoder.x1.weight` ... `lrp_transforms.9.4.bias`, `entropy_bottleneck.quantiles`), identical forward signature and
return values, so a reference checkpoint loads with `load_state_dict(..., strict=False)`.

What runs where: masked window attention, GDN / IGDN, the alpha pyramid, every rounding step and (in inference) the
convolutions -- tcgen05 implicit GEMMs chained through fp16 hi / lo planes, with GELU / ReLU, residual adds, the wrapper's
gate, the slice loop's quantisation and lrp update as epilogues (csrc/conv_tc.cu) -- are this package's sm_100a kernels;
the 3-channel ends (x1, x4, the DSE 1x1s) and everything that records autograd history are torch (cuDNN).  The entropy models are restated from CompressAI's published definitions (factorised prior of Balle et al. 2018,
Gaussian conditional with scale lower bound 0.11 and likelihood lower bound 1e-9) only to produce the bpp terms of the
forward; they are not part of the parity contract (DESIGN.md section 3, "parity unpinned").
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import quant
from . import rgba8 as rgba8_mod
from .layers.GDN import GDN
from .layers.Masked_Attention import Win_noShift_Attention, conv3x3
from .layers.conv import ACT_ADD2, ACT_LRP, ACT_QUANT, ACT_RELU, Conv2d, ConvStack, ConvTranspose2d, SplitAct
from .layers.SupplyMask import SupplyMaskToTransform, alpha_pyramid


def _conv(cin, cout, k, stride=1):
    return Conv2d(cin, cout, k, stride=stride, padding=k // 2)


def _deconv5(cin, cout):
    return ConvTranspose2d(cin, cout, 5, stride=2, padding=2, output_padding=1)


def _subpel(cin, cout, r=2):
    return nn.Sequential(Conv2d(cin, cout * r * r, 3, padding=1), nn.PixelShuffle(r))


class EnhancementBlock(nn.Module):
    """layers/TransformRGB.py:16-28"""

    def __init__(self, n=32):
        super().__init__()
        self.conv1 = Conv2d(n, n, 3, padding=1)
        self.relu = nn.ReLU(inplace=True)
        self.conv2 = Conv2d(n, n, 3, padding=1)

    def forward(self, x, **kw):
        if self.conv1.input_ps(x) is None:
            return self.conv2(self.conv1(x, act=ACT_RELU), residual=x)
        # conv1's output exists only as the planes conv2 reads; x may be a SplitAct carrying its dense tensor
        return self.conv2(self.conv1(x, act=ACT_RELU, emit_ps=1, want_dense=False),
                          residual=x.dense if isinstance(x, SplitAct) else x, **kw)


class DSE(nn.Module):
    """layers/TransformRGB.py:30-49"""

    def __init__(self, n=32):
        super().__init__()
        self.input_conv = Conv2d(3, n, 1)
        self.enh1, self.enh2, self.enh3 = EnhancementBlock(n), EnhancementBlock(n), EnhancementBlock(n)
        self.output_conv = Conv2d(n, 3, 1)

    def forward(self, x):
        if self.input_conv.input_ps(x) is None:
            first = self.input_conv(x)
            t = self.enh3(self.enh2(self.enh1(first)))
            return self.output_conv(t + first, residual=x)
        # one chain: every intermediate that only feeds a convolution exists as planes alone; the last enhancement block's
        # second convolution adds its identity AND the skip `first`, and hands planes to the output convolution
        first = self.input_conv(x, emit_ps=1)
        t = self.enh2(self.enh1(first, emit_ps=1), emit_ps=1)
        h = self.enh3.conv1(t, act=ACT_RELU, emit_ps=1, want_dense=False)
        s = self.enh3.conv2(h, act=ACT_ADD2, residual=t.dense, aux=first.dense, emit_ps=1, want_dense=False)
        return self.output_conv(s, residual=x)


def _gdn_into(gdn, x, consumer):
    """gdn(x) for the convolution `consumer`: as the fp16 hi / lo planes it reads when both take their B200 paths
    (gdn_forward_planes: no fp32 result, no split launch), else the dense tensor"""
    ps = consumer.input_ps(x) if torch.is_tensor(x) and x.dim() == 4 and x.shape[1] == consumer.in_channels else None
    return gdn.request_planes(ps)(x) if ps else gdn(x)


def _attention_into(attention, x, mask, consumer):
    """the attention wrapper for the convolution `consumer`: its gate epilogue writes the consumer's input planes when the
    wrapper runs as the convolution chain and the consumer takes the kernel, else the dense tensor"""
    ps = consumer.input_ps(x) if torch.is_tensor(x) and x.dim() == 4 and x.shape[1] == consumer.in_channels else None
    if ps and attention.conv_a[0].conv[0].input_ps(x) is not None:
        return attention.request_planes(ps)(x, mask)
    return attention(x, mask)


class Analysis_transform(nn.Module):
    """layers/TransformRGB.py:52-75"""

    def __init__(self, N=192, M=320):
        super().__init__()
        self.x1 = _conv(3, N, 5, 2)
        self.gdn1 = GDN(N)
        self.x2 = _conv(N, N, 5, 2)
        self.gdn2 = GDN(N)
        self.attention1 = Win_noShift_Attention(dim=N, num_heads=8, window_size=8, shift_size=4)
        self.x3 = _conv(N, N, 5, 2)
        self.gdn3 = GDN(N)
        self.x4 = Conv2d(N, M, 1)
        self.attention2 = Win_noShift_Attention(dim=M, num_heads=8, window_size=4, shift_size=2)

    def forward(self, input, mask, me1, me2, me3, me4):
        # a GDN whose only consumer is a convolution on the kernel writes that convolution's input planes directly
        y = _gdn_into(self.gdn1, self.x1(input), self.x2)
        y = self.gdn2(self.x2(y))
        y = _attention_into(self.attention1, y, me2, self.x3)
        y = _gdn_into(self.gdn3, self.x3(y), self.x4)
        return self.attention2(self.x4(y), me3)


class Synthesis_transform(nn.Module):
    """layers/TransformRGB.py:77-100"""

    def __init__(self, N=196, M=320):
        super().__init__()
        self.attention1 = Win_noShift_Attention(dim=M, num_heads=8, window_size=4, shift_size=2)
        self.x1 = Conv2d(M, N, 1)
        self.igdn1 = GDN(N, inverse=True)
        self.x2 = _deconv5(N, N)
        self.igdn2 = GDN(N, inverse=True)
        self.attention2 = Win_noShift_Attention(N, num_heads=8, window_size=8, shift_size=4)
        self.x3 = _deconv5(N, N)
        self.igdn3 = GDN(N, inverse=True)
        self.x4 = _deconv5(N, 3)
        self.dse = DSE(32)

    def forward(self, input, reconmask, md1, md2, md3, md4):
        y = _attention_into(self.attention1, input, md3, self.x1)
        y = _gdn_into(self.igdn1, self.x1(y), self.x2)
        y = self.igdn2(self.x2(y))
        y = _attention_into(self.attention2, y, md2, self.x3)
        y = _gdn_into(self.igdn3, self.x3(y), self.x4)
        return self.dse(self.x4(y))


class EntropyBottleneck(nn.Module):
    """Factorised prior (CompressAI's EntropyBottleneck, filters (3, 3, 3, 3), init_scale 10): parameter names and
    shapes of the real class so that its checkpoints load; `likelihood` evaluates the learned density on z_hat."""

    def __init__(self, channels, filters=(3, 3, 3, 3), init_scale=10.0):
        super().__init__()
        self.channels = channels
        f = (1,) + tuple(filters) + (1,)
        scale = init_scale ** (1.0 / (len(filters) + 1))
        for i in range(len(filters) + 1):
            init = math.log(math.expm1(1.0 / scale / f[i + 1]))
            self.register_parameter(f"_matrix{i:d}", nn.Parameter(torch.full((channels, f[i + 1], f[i]), init)))
            self.register_parameter(f"_bias{i:d}", nn.Parameter(torch.rand(channels, f[i + 1], 1) - 0.5))
            if i < len(filters):
                self.register_parameter(f"_factor{i:d}", nn.Parameter(torch.zeros(channels, f[i + 1], 1)))
        self.nlayers = len(filters) + 1
        self.quantiles = nn.Parameter(torch.tensor([-init_scale, 0.0, init_scale]).repeat(channels, 1, 1))

    def _get_medians(self):
        return self.quantiles[:, :, 1:2].detach().reshape(1, -1, 1, 1)

    def _logits_cumulative(self, v):
        for i in range(self.nlayers):
            v = torch.matmul(F.softplus(getattr(self, f"_matrix{i:d}")), v) + getattr(self, f"_bias{i:d}")
            if i < self.nlayers - 1:
                v = v + torch.tanh(getattr(self, f"_factor{i:d}")) * torch.tanh(v)
        return v

    @torch.no_grad()
    def update(self):
        """quantised CDF of every channel's learned density over [median - minima, median + maxima] (CompressAI's
        EntropyBottleneck.update); the tables live on the host, where the coder runs"""
        from . import entropy
        q = self.quantiles.detach().float()
        medians = q[:, 0, 1]
        minima = torch.ceil(medians - q[:, 0, 0]).clamp(min=0).int()
        maxima = torch.ceil(q[:, 0, 2] - medians).clamp(min=0).int()
        length = (maxima + minima + 1).tolist()
        samples = (medians - minima)[:, None, None] + torch.arange(max(length), device=q.device)[None, None, :]
        lo, up = self._logits_cumulative(samples - 0.5), self._logits_cumulative(samples + 0.5)
        sign = -torch.sign(lo + up)
        pmf = torch.abs(torch.sigmoid(sign * up) - torch.sigmoid(sign * lo))[:, 0, :].double().cpu().numpy()
        lens = torch.tensor(length)
        tail = (torch.sigmoid(lo[:, 0, 0]) + torch.sigmoid(-up[:, 0, :].gather(1, (lens - 1).to(q.device)[:, None])[:, 0]))
        self._table = entropy.CdfTable(pmf, tail.double().cpu().numpy(), length, (-minima).tolist())
        return True

    def _symbols(self, z):
        return torch.round(z - self._get_medians()).to(torch.int32)

    def _indexes(self, B, H, W, device=None):
        """the table index of every element: its channel"""
        C = self.channels
        return torch.arange(C, dtype=torch.int32, device=device).view(1, C, 1).expand(B, C, H * W).reshape(B, -1)

    @torch.no_grad()
    def compress(self, z, coder="host", lanes=None):
        """one string per image: the channel is the table index (models/AutoEncoderRGB_Journal.py:319).  coder="host": the
        host rANS coder; "device": the lane-interleaved format coded on the GPU (`lanes` lanes, entropy.default_lanes if
        None)"""
        if getattr(self, "_table", None) is None:
            self.update()
        B, C, H, W = z.shape
        if coder == "device":
            return self._table.encode_lanes(self._symbols(z).reshape(B, -1), self._indexes(B, H, W, z.device), lanes).strings()
        if coder != "host":
            raise ValueError(f"coder must be 'host' or 'device' (got {coder!r})")
        sym = self._symbols(z).cpu().numpy()
        idx = self._indexes(1, H, W)[0].numpy()
        return [self._table.encode(sym[b], idx) for b in range(B)]

    @torch.no_grad()
    def decompress(self, strings, size):
        """(:320, :372): symbols + medians; the format of the strings picks the decoder"""
        from . import entropy
        if getattr(self, "_table", None) is None:
            self.update()
        if entropy.stream_format(strings) == "device":
            streams = entropy.LaneStreams([strings], self.quantiles.device)
            z_hat = self._decode_lanes(streams.decoder(self._table, 0), size)
            streams.check()
            return z_hat
        C, (H, W) = self.channels, size
        idx = self._indexes(1, H, W)[0].numpy()
        sym = [torch.from_numpy(self._table.decoder(st).decode(idx)).view(1, C, H, W) for st in strings]
        dev = self.quantiles.device
        return torch.cat(sym, 0).to(dev).float() + self._get_medians()

    def _decode_lanes(self, decoder, size):
        """z_hat from a LaneDecoder over its strings, on the GPU; its LaneStreams.check() is the caller's"""
        B, (H, W) = decoder.count, size
        sym = decoder.decode(self._indexes(B, H, W, self.quantiles.device).contiguous())
        return sym.view(B, self.channels, H, W).float() + self._get_medians()

    def likelihood(self, z_hat):
        B, C = z_hat.shape[:2]
        v = z_hat.transpose(0, 1).reshape(C, 1, -1)
        lo, up = self._logits_cumulative(v - 0.5), self._logits_cumulative(v + 0.5)
        sign = -torch.sign(lo + up).detach()
        lik = torch.abs(torch.sigmoid(sign * up) - torch.sigmoid(sign * lo)).clamp_min(1e-9)
        return lik.reshape(C, B, *z_hat.shape[2:]).transpose(0, 1)


class GaussianConditional(nn.Module):
    """Gaussian conditional (CompressAI: scale_bound 0.11, likelihood_bound 1e-9) evaluated on y - mu."""

    def __init__(self, scale_table=None):
        super().__init__()
        self.scale_table, self._table = None, None
        self._scale_table_copies = {}

    def update_scale_table(self, scale_table, force=False):
        """one quantised Gaussian CDF per scale level (CompressAI's GaussianConditional.update_scale_table + update)"""
        from . import entropy
        if self._table is not None and not force:
            return False
        self.scale_table = torch.as_tensor(scale_table, dtype=torch.float32).clone()
        self._scale_table_copies = {}
        self._table = entropy.gaussian_table(self.scale_table)
        return True

    def build_indexes(self, scales):
        """the scale table is copied to the scales' device once (a copy per call would synchronise every slice)"""
        from . import entropy
        if scales.device not in self._scale_table_copies:
            self._scale_table_copies[scales.device] = self.scale_table.to(scales.device)
        return entropy.build_indexes(scales, self._scale_table_copies[scales.device])

    @staticmethod
    def likelihood(y, scales, means):
        v = torch.abs(y - means)
        s = torch.clamp_min(scales, 0.11)
        c = 2 ** -0.5
        upper = 0.5 * torch.erfc(-c * (0.5 - v) / s)
        lower = 0.5 * torch.erfc(-c * (-0.5 - v) / s)
        return (upper - lower).clamp_min(1e-9)


def reconstruct_error(input, output, input_mask, output_mask=None):
    """models/AutoEncoderRGB_Journal.py:36-64: squared error over the pixels whose input alpha is > 0."""
    m = (input_mask.expand(-1, 3, -1, -1) > 0.0).float()
    se = F.mse_loss(input * m, output * m, reduction="none").sum(dim=(1, 2, 3))
    return torch.mean(se / torch.clamp(m.sum(dim=(1, 2, 3)), min=1))


def _bits(lik):
    return torch.sum(torch.clamp(-1.0 * torch.log(lik + 1e-10) / math.log(2.0), 0, 50))


class AutoEncoder(nn.Module):
    """models/AutoEncoderRGB_Journal.py:124-297 (N = 192, M = 80, 10 slices, 5 support slices)."""

    def __init__(self):
        super().__init__()
        self.N, self.M = 192, 80
        N, M = self.N, self.M
        self.Encoder = Analysis_transform(N, M)
        self.Decoder = Synthesis_transform(N, M)
        self.EncMakeMask = SupplyMaskToTransform()
        self.DecMakeMask = SupplyMaskToTransform()
        self.num_slices, self.max_support_slices = 10, 5
        g = nn.GELU
        self.h_a = ConvStack(conv3x3(M, 320, stride=2), g(), conv3x3(320, 288), g(), conv3x3(288, 256, stride=2), g(),
                                 conv3x3(256, 224), g(), conv3x3(224, 192, stride=2))

        def hyper_s():
            return ConvStack(_subpel(192, 192), g(), conv3x3(192, 224), g(), _subpel(224, 256), g(),
                                 conv3x3(256, 288), g(), _subpel(288, M))

        self.h_mean_s, self.h_scale_s = hyper_s(), hyper_s()
        sl = M // self.num_slices

        def cc(cin):
            return ConvStack(_conv(cin, 224, 3), g(), _conv(224, 128, 3), g(), _conv(128, sl, 3))

        self.cc_mean_transforms = nn.ModuleList(cc(M + sl * min(i, 5)) for i in range(self.num_slices))
        self.cc_scale_transforms = nn.ModuleList(cc(M + sl * min(i, 5)) for i in range(self.num_slices))
        self.lrp_transforms = nn.ModuleList(cc(M + sl * min(i + 1, 6)) for i in range(self.num_slices))
        self.entropy_bottleneck = EntropyBottleneck(192)
        self.gaussian_conditional = GaussianConditional(None)

    # ------------------------------------------------------------------------------------------------ pieces
    def hyper(self, y):
        """z, z_hat, latent means / scales   (:223-232)"""
        z = self.h_a(y)
        z_hat = quant.quantize_offset(z, self.entropy_bottleneck._get_medians())
        return z, z_hat, self.h_mean_s(z_hat), self.h_scale_s(z_hat)

    def slice_loop(self, y, latent_means, latent_scales, want_scales=True):
        """the channel-conditional loop (:240-266).  Inference: the support tensors are assembled once -- slice i's y_hat
        is rounded straight into its channel range of a (B, M + 6 sl, H, W) buffer whose prefixes are the `torch.cat`s of
        the reference, so no concatenation kernel runs.  With autograd recording (training) the buffer trick is not
        allowed (convolutions keep views of it for their backward), and the supports are concatenated as in the reference."""
        B, M, H, W = y.shape
        sl, ms = M // self.num_slices, self.max_support_slices
        in_place = not (torch.is_grad_enabled() and (y.requires_grad or latent_means.requires_grad))
        if in_place and self.cc_mean_transforms[0][0].input_ps(latent_means) is not None:
            return self._slice_loop_fused(y, latent_means, latent_scales, want_scales)
        if in_place:
            return self._slice_loop_in_place(y, latent_means, latent_scales, want_scales)
        y_hat_slices, mus, scales = [], [], []
        for i, y_slice in enumerate(y.chunk(self.num_slices, 1)):
            support = y_hat_slices[:ms]
            mean_support = torch.cat([latent_means] + support, dim=1)
            mu = self.cc_mean_transforms[i](mean_support)[:, :, :H, :W]
            if want_scales:
                scales.append(self.cc_scale_transforms[i](torch.cat([latent_scales] + support, dim=1))[:, :, :H, :W])
            y_hat = quant.quantize_offset(y_slice, mu)
            y_hat = quant.lrp_add(y_hat, self.lrp_transforms[i](torch.cat([mean_support, y_hat], dim=1)))
            y_hat_slices.append(y_hat)
            mus.append(mu)
        return (torch.cat(y_hat_slices, 1), torch.cat(mus, 1), torch.cat(scales, 1) if want_scales else None)

    def _slice_loop_fused(self, y, latent_means, latent_scales, want_scales):
        """inference on the B200 convolution kernel: no elementwise launch and no concatenation in the loop.
        * the supports live as fp16 hi / lo planes [latent means | y_hat_0 .. y_hat_4 | scratch slice] (and the same with
          the latent scales in front); a convolution reads a channel PREFIX of them -- one of the reference's torch.cats;
        * the last convolution of cc_mean_transforms[i] quantises in its epilogue: mu goes to its slice of `means`,
          ste_round(y_i - mu) + mu (:257) as fp32 for the lrp step and as planes into the slot behind the supports;
        * the last convolution of lrp_transforms[i] adds 0.5 tanh(lrp) (:262-264) in its epilogue, writes y_hat_i into its
          slice of the result and, for i < 5, its planes into the support slot."""
        from .layers.conv import split_into
        B, M, H, W = y.shape
        sl, ms = M // self.num_slices, self.max_support_slices
        dev = y.device
        mean_sup = split_into(latent_means, SplitAct.empty(B, M, H, W, 1, dev, channels=M + (ms + 1) * sl))
        scale_sup = split_into(latent_scales, SplitAct.empty(B, M, H, W, 1, dev, channels=M + ms * sl)) if want_scales else None
        y_hat_all, means = torch.empty_like(y), torch.empty_like(y)
        scales = torch.empty_like(y) if want_scales else None
        yq = torch.empty(B, sl, H, W, device=dev, dtype=y.dtype)
        for i in range(self.num_slices):
            k = min(i, ms)
            lo, hi = i * sl, (i + 1) * sl
            slot = M + k * sl
            self.cc_mean_transforms[i](mean_sup.prefix(slot), final_act=ACT_QUANT, aux=y[:, lo:hi], out=yq,
                                       out2=means[:, lo:hi], emit_into=(mean_sup, slot))
            if want_scales:
                self.cc_scale_transforms[i](scale_sup.prefix(slot), out=scales[:, lo:hi])
            self.lrp_transforms[i](mean_sup.prefix(slot + sl), final_act=ACT_LRP, aux=yq, out=y_hat_all[:, lo:hi],
                                   emit_into=(mean_sup, slot) if i < ms else None)
            if i < ms and want_scales:                   # the same planes for the scale branch's supports
                scale_sup.hi[..., slot:slot + sl] = mean_sup.hi[..., slot:slot + sl]
                scale_sup.lo[..., slot:slot + sl] = mean_sup.lo[..., slot:slot + sl]
        return y_hat_all, means, scales

    def _slice_loop_in_place(self, y, latent_means, latent_scales, want_scales):
        B, M, H, W = y.shape
        sl, ms = M // self.num_slices, self.max_support_slices
        # mean_sup = [latent means | y_hat_0 .. y_hat_4 | scratch slice]; every prefix is one of the reference's cats
        mean_sup = torch.empty(B, M + (ms + 1) * sl, H, W, device=y.device, dtype=y.dtype)
        mean_sup[:, :M] = latent_means
        scale_sup = None
        if want_scales:
            scale_sup = torch.empty(B, M + ms * sl, H, W, device=y.device, dtype=y.dtype)
            scale_sup[:, :M] = latent_scales
        y_hat_all = torch.empty_like(y)
        mus, scales = [], []
        for i, y_slice in enumerate(y.chunk(self.num_slices, 1)):
            k = min(i, ms)
            mu = self.cc_mean_transforms[i](mean_sup[:, :M + k * sl])[:, :, :H, :W]
            if want_scales:
                scales.append(self.cc_scale_transforms[i](scale_sup[:, :M + k * sl])[:, :, :H, :W])
            # ste_round(y - mu) + mu lands in the slot right behind the supports: lrp support = that prefix
            slot = mean_sup[:, M + k * sl:M + (k + 1) * sl]
            quant.quantize_offset(y_slice, mu, out=slot)
            lrp = self.lrp_transforms[i](mean_sup[:, :M + (k + 1) * sl])
            y_hat = quant.lrp_add(slot, lrp, out=y_hat_all[:, i * sl:(i + 1) * sl])
            if i < ms:                                   # becomes a support slice of the later ones
                mean_sup[:, M + i * sl:M + (i + 1) * sl] = y_hat
                if want_scales:
                    scale_sup[:, M + i * sl:M + (i + 1) * sl] = y_hat
            mus.append(mu)
        return y_hat_all, torch.cat(mus, 1), torch.cat(scales, 1) if want_scales else None

    # ------------------------------------------------------------------------------------------------ bitstream
    def update(self, scale_table=None, force=False):
        """models/AutoEncoderRGB_Journal.py:306-311"""
        from . import entropy
        updated = self.gaussian_conditional.update_scale_table(entropy.get_scale_table() if scale_table is None else scale_table,
                                                               force=force)
        if force or getattr(self.entropy_bottleneck, "_table", None) is None:
            updated |= self.entropy_bottleneck.update()
        return updated

    @torch.no_grad()
    def compress(self, input, mask, coder="host", lanes=None):
        """models/AutoEncoderRGB_Journal.py:312-368.  The device side is the forward's own pieces (analysis, hyperprior,
        fused slice loop: one pass gives every slice's mu, scale and y_hat); one string per image (for a batch of one this
        is the reference's structure; the reference puts a whole batch into one string and can only decompress batch 1).
        coder="host": symbols and table indexes of all slices go to the host in ONE copy and the rANS coder runs there
        (csrc/rans.cu).  coder="device": the lane-interleaved format (DESIGN.md 4.7), coded on the GPU with `lanes` lanes
        per string (entropy.default_lanes of the message if None); only the finished strings cross to the host."""
        if coder not in ("host", "device"):
            raise ValueError(f"coder must be 'host' or 'device' (got {coder!r})")
        self.update()
        _, me = alpha_pyramid(mask, 3)
        y = self.Encoder(input, mask, None, me[1], me[2], None)
        z = self.h_a(y)
        eb = self.entropy_bottleneck
        if coder == "device":
            # z_hat is what the decoder will reconstruct from the z strings: their symbols + the medians
            B, _, Hz, Wz = z.shape
            z_sym = eb._symbols(z)
            z_job = eb._table.encode_lanes(z_sym.reshape(B, -1), eb._indexes(B, Hz, Wz, z.device), lanes)
            z_hat = z_sym.float() + eb._get_medians()
        else:
            z_strings = eb.compress(z)
            z_hat = eb.decompress(z_strings, z.shape[-2:])
        latent_scales, latent_means = self.h_scale_s(z_hat), self.h_mean_s(z_hat)
        _, means, scales = self.slice_loop(y, latent_means, latent_scales)
        symbols = torch.round(y - means).to(torch.int32)                       # quantize(y, "symbols", mu)   (:347)
        indexes = self.gaussian_conditional.build_indexes(scales)
        table = self.gaussian_conditional._table
        if coder == "device":
            B = y.shape[0]
            y_job = table.encode_lanes(symbols.reshape(B, -1), indexes.reshape(B, -1), lanes)
            return {"strings": [y_job.strings(), z_job.strings()], "shape": z.shape[-2:]}
        symbols, indexes = symbols.cpu().numpy(), indexes.cpu().numpy()
        y_strings = [table.encode(symbols[b], indexes[b]) for b in range(y.shape[0])]
        return {"strings": [y_strings, z_strings], "shape": z.shape[-2:]}

    @torch.no_grad()
    def decompress(self, strings, shape, mask):
        """models/AutoEncoderRGB_Journal.py:370-415: slice by slice -- mu and scale of slice i need the decoded slices < i --
        with the same kernels as the encoder, so the tables' indexes and the reconstruction are bit-identical to its.
        The strings' format picks the decoder: host-format strings are decoded on the host, slice by slice; lane-format
        strings are staged on the GPU in one copy and decoded there, with one synchronisation (the status check) in all."""
        x_hat, streams = self._decode(strings, shape, mask)
        x_hat = x_hat.clamp_(0, 1)
        if streams is not None:
            streams.check()
        return {"x_hat": x_hat}

    def _decode(self, strings, shape, mask):
        """decompress up to the synthesis transform: (unclamped x_hat, the LaneStreams whose check() is the caller's, or
        None for host-format strings)"""
        from . import entropy
        from .layers.conv import split_into
        self.update()
        eb, table = self.entropy_bottleneck, self.gaussian_conditional._table
        streams = None
        if entropy.stream_format(list(strings[0]) + list(strings[1])) == "device":
            streams = entropy.LaneStreams([strings[1], strings[0]], eb.quantiles.device)
            z_hat = eb._decode_lanes(streams.decoder(eb._table, 0), shape)
            y_decoder = streams.decoder(table, 1)
        else:
            z_hat = eb.decompress(strings[1], shape)
            decoders = [table.decoder(st) for st in strings[0]]
        latent_scales, latent_means = self.h_scale_s(z_hat), self.h_mean_s(z_hat)
        B, M, H, W = latent_means.shape
        sl, ms, dev = M // self.num_slices, self.max_support_slices, latent_means.device
        fused = self.cc_mean_transforms[0][0].input_ps(latent_means) is not None
        if fused:
            mean_sup = split_into(latent_means, SplitAct.empty(B, M, H, W, 1, dev, channels=M + (ms + 1) * sl))
            scale_sup = split_into(latent_scales, SplitAct.empty(B, M, H, W, 1, dev, channels=M + ms * sl))
        y_hat_slices = []
        for i in range(self.num_slices):
            k = min(i, ms)
            slot = M + k * sl
            if fused:
                mu = self.cc_mean_transforms[i](mean_sup.prefix(slot))
                scale = self.cc_scale_transforms[i](scale_sup.prefix(slot))
            else:
                support = y_hat_slices[:ms]
                mu = self.cc_mean_transforms[i](torch.cat([latent_means] + support, 1))
                scale = self.cc_scale_transforms[i](torch.cat([latent_scales] + support, 1))
            idx = self.gaussian_conditional.build_indexes(scale)
            if streams is not None:
                sym = y_decoder.decode(idx.reshape(B, -1)).view(B, sl, H, W)
            else:
                idx = idx.cpu().numpy()
                sym = torch.from_numpy(np.stack([decoders[b].decode(idx[b]) for b in range(B)])).view(B, sl, H, W)
            y_hat = sym.to(dev).float() + mu                                   # dequantize(rv, mu)   (:395)
            if fused:
                split_into(y_hat, mean_sup, slot)
                lrp = self.lrp_transforms[i](mean_sup.prefix(slot + sl), final_act=ACT_LRP, aux=y_hat, out=y_hat,
                                             emit_into=(mean_sup, slot) if i < ms else None)
                if i < ms:
                    scale_sup.hi[..., slot:slot + sl] = mean_sup.hi[..., slot:slot + sl]
                    scale_sup.lo[..., slot:slot + sl] = mean_sup.lo[..., slot:slot + sl]
            else:
                y_hat = quant.lrp_add(y_hat, self.lrp_transforms[i](torch.cat([latent_means] + y_hat_slices[:ms] + [y_hat], 1)))
            y_hat_slices.append(y_hat)
        _, md = alpha_pyramid(mask, 3)
        return self.Decoder(torch.cat(y_hat_slices, 1), mask, None, md[1], md[2], None), streams

    @torch.no_grad()
    def compress_rgba8(self, rgba8, coder="host", lanes=None):
        """compress for 8-bit RGBA of any size: uint8 (B, H, W, 4) or (H, W, 4), on the GPU or the host (copied once).
        The image is converted on the device to the planes the model was trained on (a / 255, colour premultiplied by the
        binarised alpha; csrc/rgba8.cu) and padded at the bottom and right with transparent pixels to multiples of 64, then
        compressed as `compress` does; the stream format is unchanged.  Returns {"strings", "shape", "size": (H, W)}."""
        return self._compress_rgba(rgba8, torch.uint8, None, coder, lanes)

    @torch.no_grad()
    def decompress_rgba8(self, strings, shape, alpha8):
        """decompress to uint8 (B, H, W, 4).  alpha8: uint8 (B, H, W) or (H, W), the images' alpha (the decoder takes it as
        `decompress` takes the mask); it gives the original size, and shape must be (ceil(H / 64), ceil(W / 64)).  Alpha is
        copied through; RGB = rint(clamp(x_hat, 0, 1) * 255) where alpha > 0, else 0, cropped to H x W in one launch."""
        return self._decompress_rgba(strings, shape, alpha8, torch.uint8, False)

    @torch.no_grad()
    def compress_rgba16(self, rgba16, coder="host", lanes=None):
        """compress_rgba8 for 16-bit RGBA: uint16 (B, H, W, 4) or (H, W, 4), converted with full scale 65535.  The stream
        format is the same: for 8-bit values v, rgba16 = 257 * v gives exactly compress_rgba8's strings."""
        return self._compress_rgba(rgba16, torch.uint16, None, coder, lanes)

    @torch.no_grad()
    def decompress_rgba16(self, strings, shape, alpha16):
        """decompress_rgba8 to uint16 (B, H, W, 4) given the uint16 (B, H, W) or (H, W) alpha: RGB = rint(clamp(x_hat, 0, 1)
        * 65535) where alpha > 0, else 0.  Strings from compress_rgba8, compress_rgba16 or compress decode alike."""
        return self._decompress_rgba(strings, shape, alpha16, torch.uint16, False)

    @torch.no_grad()
    def compress_tiled(self, rgba, tile=4096, coder="host", lanes=None):
        """compress uint8 or uint16 RGBA (B, H, W, 4) or (H, W, 4) of any size and any batch, on the GPU or the host
        (copied once), as independent tiles of Th x Tw = rgba8.tile_grid(H, W, tile) (DESIGN.md 4.8): tile n = (b * ty + i)
        * tx + j covers rows i * Th.. and columns j * Tw.. of image b, padded with transparent pixels past the image.  Each
        tile is coded exactly as compress_rgba8 / 16 codes that crop padded to Th x Tw; the passes take as many tiles as
        one forward can index (rgba8.chunk_tiles).  Returns {"strings": [y strings, z strings] of B * ty * tx tiles each in
        tile order, "shape": (Th / 64, Tw / 64), "size": (H, W), "grid": (ty, tx)}.  With tile >= the padded image the grid
        is 1 x 1 and the strings are compress_rgba8 / 16's."""
        rgba8_mod.depth(rgba, "rgba")
        return self._compress_rgba(rgba, rgba.dtype, tile, coder, lanes)

    @torch.no_grad()
    def decompress_tiled(self, strings, shape, alpha):
        """decompress compress_tiled's strings (or compress_rgba8 / 16's, a 1 x 1 grid) to (B, H, W, 4) of the alpha's
        dtype, given the images' uint8 or uint16 (B, H, W) or (H, W) alpha: the grid follows from its size and the tile
        shape; each tile decodes as decompress_rgba8 / 16 decodes it, and the tiles are stitched into one output."""
        rgba8_mod.depth(alpha, "alpha")
        return self._decompress_rgba(strings, shape, alpha, alpha.dtype, True)

    def _compress_rgba(self, rgba, dtype, tile, coder, lanes):
        """compress in tiles of tile_grid(H, W, tile), or of the padded image (tile None: the size guard applies), a chunk
        of tiles per forward pass"""
        if coder not in ("host", "device"):
            raise ValueError(f"coder must be 'host' or 'device' (got {coder!r})")
        t = rgba8_mod.as_batch(rgba, (4,), f"rgba{8 * dtype.itemsize}", dtype)
        B, H, W, _ = t.shape
        if tile is None:
            rgba8_mod._check_size(B, H, W)
            Th, Tw, ty, tx = rgba8_mod.padded(H), rgba8_mod.padded(W), 1, 1
        else:
            Th, Tw, ty, tx = rgba8_mod.tile_grid(H, W, tile)
        t = rgba8_mod.staged(t, self.entropy_bottleneck.quantiles.device)
        n, per = B * ty * tx, rgba8_mod.chunk_tiles(Th, Tw)
        strings = [[], []]
        for first in range(0, max(n, 1), per):
            image, alpha = rgba8_mod.ingest_tiles(t, (Th, Tw), first, min(per, n - first))
            out = self.compress(image, alpha, coder=coder, lanes=lanes)
            strings[0] += out["strings"][0]
            strings[1] += out["strings"][1]
        out["strings"], out["size"] = strings, (H, W)
        if tile is not None:
            out["shape"], out["grid"] = (Th // rgba8_mod.PAD, Tw // rgba8_mod.PAD), (ty, tx)
        return out

    def _decompress_rgba(self, strings, shape, alpha_in, dtype, tiled):
        a = rgba8_mod.as_batch(alpha_in.unsqueeze(-1) if isinstance(alpha_in, torch.Tensor) else alpha_in, (1,),
                               f"alpha{8 * dtype.itemsize}", dtype)
        B, H, W, _ = a.shape
        want = (rgba8_mod.padded(H) // rgba8_mod.PAD, rgba8_mod.padded(W) // rgba8_mod.PAD)
        if tiled:
            Th, Tw, ty, tx = rgba8_mod.tiles_of(H, W, shape)
        elif tuple(int(v) for v in shape) != want:
            raise ValueError(f"shape {tuple(shape)} does not fit a {H} x {W} alpha: expected {want}")
        else:
            Th, Tw, ty, tx = want[0] * rgba8_mod.PAD, want[1] * rgba8_mod.PAD, 1, 1
        n = B * ty * tx
        if len(strings) != 2 or len(strings[0]) != n or len(strings[1]) != n:
            raise ValueError(f"expected [y strings, z strings] of {n} {'tiles' if tiled else 'images'} each")
        if not tiled:
            rgba8_mod._check_size(B, H, W)
        a = rgba8_mod.staged(a, self.entropy_bottleneck.quantiles.device)
        out = torch.empty(B, H, W, 4, dtype=dtype, device=a.device)
        per = rgba8_mod.chunk_tiles(Th, Tw)
        for first in range(0, max(n, 1), per):
            count = min(per, n - first)
            _, alpha = rgba8_mod.ingest_tiles(a, (Th, Tw), first, count)
            x_hat, streams = self._decode([strings[0][first:first + count], strings[1][first:first + count]], shape, alpha)
            rgba8_mod.egress_tiles(x_hat, a.view(B, H, W), out, first)
            if streams is not None:
                streams.check()
        return out

    def detail(self, input, mask, reconmask, me2=None, me3=None):
        """every tensor of the forward the parity tests look at"""
        if me2 is None:
            _, me = alpha_pyramid(mask, 3)
            me2, me3 = me[1], me[2]
        reconmask, md = alpha_pyramid(reconmask, 3, quant_levels=255)     # (:212-215) in the pyramid's first launch
        y = self.Encoder(input, reconmask, None, me2, me3, None)
        z, z_hat, latent_means, latent_scales = self.hyper(y)
        y_hat, means, scales = self.slice_loop(y, latent_means, latent_scales)
        x_hat = self.Decoder(y_hat, reconmask, None, md[1], md[2], None)
        return dict(y=y, z=z, z_hat=z_hat, y_hat=y_hat, means=means, scales=scales, x_hat=x_hat)

    def _rate_terms_fused(self, input, mask, r):
        """mse, y bpp, z bpp, total bpp in four launches of csrc/rate.cu (rate_forward) -- inference on CUDA with the
        factorised prior's standard filters; None when the call has to stay with the torch expressions below"""
        eb = self.entropy_bottleneck
        if torch.is_grad_enabled() or not input.is_cuda or eb.nlayers != 5 or tuple(eb._matrix1.shape[1:]) != (3, 3):
            return None
        from . import _abi
        import ctypes
        lib = _abi.load()
        y, scales, means, z_hat, x_hat = (r[k].contiguous() for k in ("y", "scales", "means", "z_hat", "x_hat"))
        inp, m = input.contiguous(), mask.contiguous()
        if any(t.dtype != torch.float32 for t in (y, scales, means, z_hat, x_hat, inp, m)) or m.numel() != inp.numel() // inp.shape[1]:
            return None
        B, C, H, W = inp.shape
        names = [f"_matrix{i}" for i in range(5)] + [f"_bias{i}" for i in range(5)] + [f"_factor{i}" for i in range(4)]
        params = [getattr(eb, n).detach().contiguous() for n in names]
        ptrs = (ctypes.c_void_p * 14)(*[p.data_ptr() for p in params])
        ws = torch.empty(int(lib.rate_workspace_bytes(B)) // 8, dtype=torch.float64, device=inp.device)
        out = torch.empty(4, dtype=torch.float32, device=inp.device)
        with torch.cuda.device(inp.device):
            _abi.check(lib.rate_forward(inp.data_ptr(), x_hat.data_ptr(), m.data_ptr(), B, C, H, W, y.data_ptr(),
                                        scales.data_ptr(), means.data_ptr(), y.numel(), z_hat.data_ptr(), ptrs,
                                        z_hat.shape[1], z_hat.shape[2] * z_hat.shape[3], ws.data_ptr(), ws.numel() * 8,
                                        out.data_ptr(), _abi.stream_handle()), "rate_forward")
        _abi.count_launches(4)
        return out

    def forward(self, input, mask, reconmask, me1, me2, me3, me4):
        r = self.detail(input, mask, reconmask, me2, me3)
        t = self._rate_terms_fused(input, mask, r)
        if t is not None:
            return r["x_hat"], t[0], t[3], t[1], t[2]
        y_bits = _bits(self.gaussian_conditional.likelihood(r["y"], r["scales"], r["means"]))
        z_bits = _bits(self.entropy_bottleneck.likelihood(r["z_hat"]))
        mse_loss = reconstruct_error(input, r["x_hat"], mask, reconmask)
        px = input.shape[0] * input.shape[2] * input.shape[3]
        total_y_bpp, total_z_bpp = y_bits / px, z_bits / px
        return r["x_hat"], mse_loss, total_y_bpp + total_z_bpp, total_y_bpp, total_z_bpp
