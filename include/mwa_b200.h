/*
 * mwa_b200.h -- C ABI of the B200-native hot path: masked window attention, GDN / IGDN, latent rounding.
 *
 * The reference (Yoshiki172/Deep-Learning-based-RGBA-Image-Compression-with-Masked-Window-based-Attention)
 * is pure Python and has no FFI; its boundary for this path is the nn.Module API of three files
 * (SURVEY.md section 8b).  Each entry point below names the reference interface it replaces
 * (paths relative to the reference root).  The Python drop-in modules in
 * `<package>/layers/` bind these symbols with ctypes (see INTEGRATION.md for the stub).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer valid on the current device;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it, never synchronise,
 *     never allocate; the caller owns all memory including workspaces;
 *   - tensors are fp32, dense, either NCHW (`channels_last == 0`) or NHWC (`channels_last == 1`);
 *   - return value: MWA_OK or a negative MWA_ERR_* code; mwa_b200_status_string() describes it.
 */
#ifndef MWA_B200_H_
#define MWA_B200_H_

#include <stdint.h>

#if defined(__GNUC__)
#define MWA_API __attribute__((visibility("default")))
#else
#define MWA_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MWA_B200_ABI_VERSION 1

enum {
    MWA_OK = 0,
    MWA_ERR_INVALID = -1,      /* bad argument (null pointer, non-positive size, shift >= window ...) */
    MWA_ERR_UNSUPPORTED = -2,  /* shape outside what the kernels cover (documented per function) */
    MWA_ERR_ALIGNMENT = -3,    /* pointer not 16-byte aligned */
    MWA_ERR_WORKSPACE = -4,    /* workspace too small */
    MWA_ERR_CUDA = -5          /* a CUDA runtime call failed (launch error) */
};

/* kernel selection.  AUTO is fp32-faithful on every shape (the reference's arithmetic is fp32 end to end; every output
 * within 1e-3 relative / 1e-4 absolute of it):
 *   C = 192, 8 x 8 windows, 6 or 8 heads, NCHW   split-precision tcgen05 kernel (every operand fp16 hi + lo, 3 MMA passes)
 *   C = 80, 4 x 4 windows, 8 heads, NCHW         plain fp32 kernel for small windows
 *   anything else                                general fp32 SIMT kernel (also what SIMT forces)
 * TCGEN05 forces the tensor-core kernel: the split-precision kernel for attention, the tcgen05 kernel for GDN;
 * MWA_ERR_UNSUPPORTED where it does not cover the shape.  Any other value is MWA_ERR_INVALID. */
enum { MWA_ALGO_AUTO = 0, MWA_ALGO_SIMT = 1, MWA_ALGO_TCGEN05 = 2 };

MWA_API int mwa_b200_abi_version(void);
MWA_API const char* mwa_b200_status_string(int status);
/* last CUDA error string recorded by a failing call on this thread ("" if none) */
MWA_API const char* mwa_b200_last_cuda_error(void);

/* ------------------------------------------------------------------------------------------------
 * GDN / IGDN      replaces  layers/GDN.py:64-94  (GDN.forward)  and  :9-23 (LowerBound, fwd part)
 *
 * gdn_prepare   : beta = max(beta_p, beta_bound)^2 - pedestal ; gamma = max(gamma_p, gamma_bound)^2 - pedestal
 *                 (layers/GDN.py:74-80) expanded into the kernel-ready parameter block `params`
 *                 (fp32 beta / gamma / gamma^T and the bf16 hi/lo UMMA operand images of gamma).
 * gdn_forward   : y[i] = x[i] * (beta[i] + sum_j gamma[i][j] * x[j]^2) ^ (-1/2)   (inverse: ^ (+1/2))
 *                 per pixel, x/y of logical shape (n_img, C, hw)  (layers/GDN.py:83-90).
 * gdn_backward  : gradients wrt x, beta_p, gamma_p incl. the LowerBound pass-through rule
 *                 (layers/GDN.py:17-23).  dbeta_p / dgamma_p are OVERWRITTEN (not accumulated).
 * Supported: 1 <= C <= 512 (SIMT); C == 192 (tcgen05).
 * ------------------------------------------------------------------------------------------------ */
MWA_API int64_t gdn_param_bytes(int C);
MWA_API int gdn_prepare(const float* beta_p, const float* gamma_p, int C, float beta_bound, float gamma_bound,
                float pedestal, void* params, int64_t params_bytes, void* stream);
MWA_API int gdn_forward(const float* x, float* y, const void* params, int64_t n_img, int C, int64_t hw, int inverse,
                int channels_last, int algo, void* stream);
/* gdn_forward_planes : the same GDN / IGDN whose consumer is a convolution of this library (layers/TransformRGB.py:55-61,
 *                 :81-88 -- gdn1 -> x2, gdn3 -> x4, igdn1 -> x2, igdn3 -> x4): y is written ONLY as the fp16 hi / lo planes
 *                 that convolution's TMA reads ([n_img][ps*ps][H/ps][W/ps][out_cstride] channels last, ps = 2 for a stride-2
 *                 consumer), bit-identical to conv_act_split of gdn_forward's y; no fp32 tensor and no split launch in
 *                 between.  x fp32 NCHW, C == 192 (tcgen05 kernel only: MWA_ERR_UNSUPPORTED otherwise). */
MWA_API int gdn_forward_planes(const float* x, void* out_hi, void* out_lo, int ps, int out_cstride, const void* params,
                       int64_t n_img, int C, int H, int W, int inverse, void* stream);
MWA_API int64_t gdn_backward_workspace_bytes(int64_t n_img, int C, int64_t hw);
MWA_API int gdn_backward(const float* x, const float* grad_y, const float* beta_p, const float* gamma_p,
                 const void* params, float beta_bound, float gamma_bound, float* grad_x, float* grad_beta_p,
                 float* grad_gamma_p, void* workspace, int64_t workspace_bytes, int64_t n_img, int C, int64_t hw,
                 int inverse, int channels_last, void* stream);

/* GEMM-composed GDN backward (what the Python layer uses for C == 192 when algo != SIMT): the three C x C contractions
 * are plain GEMMs over the pixel dimension, run by the caller with a library GEMM on the fp32 effective gamma / gamma^T
 * inside the parameter block (byte offsets from gdn_param_offset: which = 0 beta, 1 gamma [i][j], 2 gamma^T [j][i]);
 * these entry points are the hand-written stages in between, one pass over the tensors each:
 *   gdn_bwd_square   x2 = x * x
 *   (GEMM)           nb = gamma . x2          per pixel, without beta
 *   gdn_bwd_dn       n = nb + beta; dn = d loss / d n; nb is overwritten with term1 = grad_y * n^(-/+ 1/2)
 *   (GEMM)           t  = gamma^T . dn
 *   gdn_bwd_dx       grad_x = term1 + 2 x t
 *   (GEMM)           dgamma_eff = sum over pixels of dn (x2)^T
 *   gdn_bwd_finalize dbeta_eff = sum dn (dbeta_scratch: C floats), then the LowerBound / reparametrisation chain rule
 *                    (layers/GDN.py:17-23, :74-80) -> grad_beta_p, grad_gamma_p
 * Same arithmetic as gdn_backward; n = n_img * C * hw elements (multiple of 4 for the vectorised stages). */
MWA_API int64_t gdn_param_offset(int C, int which);
MWA_API int gdn_bwd_square(const float* x, float* x2, int64_t n, void* stream);
MWA_API int gdn_bwd_dn(const float* grad_y, const float* x, float* n_to_term1, const void* params, float* dn,
                       int64_t n_img, int C, int64_t hw, int inverse, int channels_last, void* stream);
MWA_API int gdn_bwd_dx(const float* term1, const float* x, const float* t, float* grad_x, int64_t n, void* stream);
MWA_API int gdn_bwd_finalize(const float* dn, const float* dgamma_eff, const float* beta_p, const float* gamma_p,
                             float beta_bound, float gamma_bound, float* grad_beta_p, float* grad_gamma_p,
                             float* dbeta_scratch, int64_t n_img, int C, int64_t hw, int channels_last, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Masked window attention   replaces  layers/masked_win_attention.py:169-251 (WinBasedAttention.forward,
 *   with its helpers window_partition :6-18, window_reverse :20-33, remove_zero_windows :35-47 and
 *   WindowAttention.forward :96-131)  and  layers/win_attention.py:153-207 (alpha == NULL).
 *
 * mwa_prepare : packs qkv.weight (3C,C), qkv.bias (3C) or NULL, proj.weight (C,C), proj.bias (C),
 *               relative_position_bias_table ((2ws-1)^2, heads) into `params`: fp32 transposes, the
 *               expanded (heads, N, N) bias (layers/masked_win_attention.py:109-112) and, where the split-precision
 *               kernel covers the shape, its fp16 hi / lo UMMA images.
 * mwa_forward : out = x + scatter(window_attention(kept windows of roll(x, -shift)))  rolled back;
 *               a window is kept iff the sum of its (shifted) alpha is != 0; alpha == NULL keeps all.
 *               x/out logical shape (B, C, H, W), alpha (B, 1, H, W); H % ws == 0 and W % ws == 0
 *               (else MWA_ERR_INVALID, the reference raises in .view); 0 <= shift < ws.
 *               `kept_count` (optional device int32, may be NULL) receives the number of kept windows.
 *               `workspace` (>= mwa_workspace_bytes(B, H, W, ws) bytes, 16-byte aligned, device) holds the keep flags
 *               and the ordered lists of kept and dropped windows of the split-precision and small-window kernels;
 *               contents are scratch.
 * Supported: ws*ws <= 64 tokens, C % heads == 0, shared memory footprint <= 227 KB (SIMT: C <= 192 at ws 8);
 *            tcgen05 (split precision): (C, heads, ws) in {(192, 8, 8), (192, 6, 8)}, NCHW.
 * ------------------------------------------------------------------------------------------------ */
MWA_API int64_t mwa_param_bytes(int C, int heads, int ws);
MWA_API int mwa_prepare(const float* qkv_w, const float* qkv_b, const float* proj_w, const float* proj_b,
                const float* bias_table, int C, int heads, int ws, float scale, void* params,
                int64_t params_bytes, void* stream);
MWA_API int64_t mwa_workspace_bytes(int B, int H, int W, int ws);
/* 1 when MWA_ALGO_AUTO has a fast fp32-faithful kernel for this configuration that reads NCHW only (the host layer then
 * hands a channels-last tensor over as NCHW instead of letting it fall to the general SIMT kernel), else 0 */
MWA_API int mwa_fast_path_needs_nchw(int C, int heads, int ws);
/* development aid: device buffer of 8192 uint64 that the split-precision attention kernel fills with clock64() totals
 * ([64,320): cycles per CTA; [320,576): tiles per CTA; [1024,5120): event trace of CTA 0, 1024 per role).  NULL switches
 * it off (the default). */
MWA_API void mwa_debug_set_timing_buffer(void* device_u64x8192);
MWA_API int mwa_forward(const float* x, const float* alpha, float* out, const void* params, int B, int C, int H, int W,
                int heads, int ws, int shift, int channels_last, int algo, int32_t* kept_count, void* workspace,
                int64_t workspace_bytes, void* stream);

/* window_attention_forward : replaces layers/masked_win_attention.py:96-131 / layers/win_attention.py:84-115
 *   (WindowAttention.forward on already-partitioned tokens): xw/out are (K, N, C) with N = ws*ws, `mask` is
 *   NULL or an additive (mask_windows, N, N) tensor applied to window k as mask[k % mask_windows]; no residual. */
MWA_API int window_attention_forward(const float* xw, const float* mask, float* out, const void* params, int64_t K,
                                     int C, int heads, int ws, int mask_windows, void* stream);

/* mwa_backward : replaces autograd through layers/masked_win_attention.py:169-251 / layers/win_attention.py:153-207.
 *   grad_x (B,C,H,W) = grad_out + d(window attention) on kept windows (dropped windows: grad_out);
 *   grad_table ((2ws-1)^2, heads) is OVERWRITTEN with the relative-position table gradient;
 *   the four token-major scratch tensors (nwin = B*(H/ws)*(W/ws) windows, N = ws*ws; rows of dropped windows are
 *   zeros) carry everything the remaining parameter gradients need as plain GEMMs / column sums over tokens:
 *     xw_tok (nwin,N,C), ao_tok (nwin,N,C), dy_tok (nwin,N,C), dqkv_tok (nwin,N,3C)
 *     grad qkv.weight = dqkv_tok^T xw_tok   grad qkv.bias = colsum(dqkv_tok)
 *     grad proj.weight = dy_tok^T ao_tok    grad proj.bias = colsum(dy_tok)
 *   qkv_w (3C,C) / proj_w (C,C) are the un-prepared fp32 weights; `params` the mwa_prepare block of the same weights.
 * window_attention_backward : same for layers/masked_win_attention.py:96-131 on (K,N,C) tokens with the optional
 *   additive (mask_windows,N,N) mask; xw / grad_out themselves play the role of xw_tok / dy_tok.
 * fp32 SIMT kernels; supported: ws*ws <= 64 tokens (multiple of 4), shared-memory footprint <= 227 KB. */
MWA_API int mwa_backward(const float* x, const float* alpha, const float* grad_out, const float* qkv_w,
                         const float* proj_w, const void* params, float* grad_x, float* grad_table, float* xw_tok,
                         float* ao_tok, float* dy_tok, float* dqkv_tok, int B, int C, int H, int W, int heads, int ws,
                         int shift, int channels_last, void* stream);
MWA_API int window_attention_backward(const float* xw, const float* mask, const float* grad_out, const float* qkv_w,
                                      const float* proj_w, const void* params, float* grad_xw, float* grad_table,
                                      float* ao_tok, float* dqkv_tok, int64_t K, int C, int heads, int ws,
                                      int mask_windows, void* stream);

/* GEMM-composed attention backward (what the Python layer uses when algo != SIMT): the token GEMMs
 *   qkv_tok = xw_tok Wqkv^T + b,  dao_tok = dy_tok Wproj,  dxw_tok = dqkv_tok Wqkv  (+ the weight-gradient GEMMs above)
 * are plain GEMMs over all tokens and run in the caller's library GEMM; these are the hand-written stages around them:
 *   mwa_bwd_gather   x, grad_out (B,C,H,W) -> xw_tok, dy_tok (nwin,N,C; zero rows for dropped windows) + keep flags (nwin)
 *   mwa_bwd_core     per window and head: softmax recompute, ao_tok, dqkv_tok (zero rows where !keep), grad_table
 *                    (OVERWRITTEN).  H > 0: image geometry (region mask from H, W, shift); H == 0: token mode with the
 *                    optional additive (mask_windows,N,N) mask and keep_flags == NULL.
 *   mwa_bwd_scatter  grad_x = grad_out + dxw_tok at the un-shifted pixel positions */
MWA_API int mwa_bwd_gather(const float* x, const float* alpha, const float* grad_out, float* xw_tok, float* dy_tok,
                           uint8_t* keep_flags, int B, int C, int H, int W, int ws, int shift, int channels_last,
                           void* stream);
MWA_API int mwa_bwd_core(const float* qkv_tok, const float* dao_tok, const void* params, const float* mask,
                         const uint8_t* keep_flags, float* ao_tok, float* dqkv_tok, float* grad_table, int64_t nwin,
                         int C, int H, int W, int heads, int ws, int shift, int mask_windows, void* stream);
MWA_API int mwa_bwd_scatter(const float* grad_out, const float* dxw_tok, float* grad_x, int B, int C, int H, int W,
                            int ws, int shift, int channels_last, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Latent rounding   replaces  models/AutoEncoderRGB_Journal.py:31-32 (ste_round; forward value) and its
 *   uses :227-229, :257, :262-264, :212-214  (= models/AutoEncoderMask_Journal.py:142-143, :255-257, :284).
 * All are elementwise over `rows` rows of `row_len` contiguous floats; row r of tensor t starts at
 * t + r * t_row_stride (lets a channel chunk of a (B,C,H,W) tensor be passed without a copy).
 *
 * round_ste_forward       : out = (rint(x) - x) + x  == rint(x), zero results are +0.0 (round-half-to-even)
 * quantize_offset_forward : out = ste_round(x - mu) + mu           mu: same shape (mu_channels == 0) or one
 *                           value per channel (mu_channels == C, row_len == C*hw, channel = (i / hw) % C)
 * lrp_add_forward         : out = y_hat + 0.5 * tanh(lrp)
 * quantize_levels_forward : out = rint(m * levels) / levels
 * ------------------------------------------------------------------------------------------------ */
MWA_API int round_ste_forward(const float* x, float* out, int64_t rows, int64_t row_len, int64_t x_row_stride,
                      int64_t out_row_stride, void* stream);
MWA_API int quantize_offset_forward(const float* x, const float* mu, float* out, int64_t rows, int64_t row_len,
                            int64_t x_row_stride, int64_t mu_row_stride, int64_t out_row_stride,
                            int mu_channels, int64_t hw, void* stream);
MWA_API int lrp_add_forward(const float* y_hat, const float* lrp, float* out, int64_t rows, int64_t row_len,
                    int64_t y_row_stride, int64_t lrp_row_stride, int64_t out_row_stride, void* stream);
MWA_API int quantize_levels_forward(const float* m, float* out, int64_t n, float levels, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Attention wrapper gate (SURVEY.md 8f, first widening step)   replaces  layers/Masked_Attention.py:186-188
 *   (Win_noShift_Attention.forward:  out = a * torch.sigmoid(b); out += identity) -- one pass instead of three kernels.
 * gate_residual_forward  : out = a * sigmoid(b) + x          n contiguous floats each (any memory format, same for all)
 * gate_residual_backward : grad_a = g * s, grad_b = g * a * s * (1 - s), s = sigmoid(b);  grad_x = g (caller's alias)
 * ------------------------------------------------------------------------------------------------ */
MWA_API int gate_residual_forward(const float* a, const float* b, const float* x, float* out, int64_t n, void* stream);
MWA_API int gate_residual_backward(const float* a, const float* b, const float* grad_out, float* grad_a, float* grad_b,
                                   int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Alpha pyramid (SURVEY.md 8f, rank 4; Appendix A "Alpha pyramid feeding a1")   replaces  layers/SupplyMask.py:7-18
 *   (SupplyMaskToTransform.forward: six cascaded AvgPool2d(3, stride 2, padding 1), count_include_pad) and, with
 *   quant_levels > 0, the decoder's mask quantisation in front of it (models/AutoEncoderRGB_Journal.py:212-214:
 *   reconmask = round(reconmask * 255) / 255).  Three levels per launch (halo recomputed in shared memory).
 * alpha  : (B, H, W) fp32 plane (the reference's (B, 1, H, W)), contiguous
 * recon  : NULL, or (B, H, W): receives the quantised plane when quant_levels > 0
 * levels : packed output, level k (1-based) = (B, H_k, W_k) at element offset alpha_pyramid_level_offset(B, H, W, k - 1),
 *          H_k = (H_{k-1} - 1) / 2 + 1; total elements = alpha_pyramid_level_offset(B, H, W, nlevels);  1 <= nlevels <= 6
 * Each output is the row-major fp32 sum of its in-range taps divided by 9 (bit-exact with torch.nn.AvgPool2d).
 * ------------------------------------------------------------------------------------------------ */
MWA_API int64_t alpha_pyramid_level_offset(int B, int H, int W, int level);
MWA_API int alpha_pyramid_forward(const float* alpha, float* recon, float* levels, int B, int H, int W, int nlevels,
                                  int quant_levels, void* stream);

/* Isolated-pixel clean-up of the decoded mask   replaces  trainRGB.py:98-111 / trainmask.py:133-146 (`constraint`) and,
 * with quant_levels > 0, the clamp + quantisation in front of it at its call site (trainRGB.py:285-287):
 *   m = round(clamp(m, 0, 1) * q) / q;  s = sum of the 8 neighbours (zero padding);
 *   out = 1 if (m == 0 && s == 8), 0 if (m > 0 && s == 0), m otherwise.      mask, out: (B, H, W) fp32, out != mask.
 * One launch, no host synchronisation (the reference's boolean-mask assignments synchronise twice). */
MWA_API int mask_constraint_forward(const float* mask, float* out, int B, int H, int W, int quant_levels, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Convolutions of the transforms (SURVEY.md 8f, the callers of the hot path)   replaces the torch.nn.Conv2d /
 *   ConvTranspose2d calls of layers/TransformRGB.py:16-100, layers/Masked_Attention.py:150-181 and
 *   models/AutoEncoderRGB_Journal.py:139-203 (F.conv2d / F.conv_transpose2d, fp32) in inference.
 *
 * kind 0: convolution, k in {1, 3, 5}, stride 1 or 2 (H, W even), padding k / 2, dilation 1, groups 1
 * kind 1: transposed convolution, k = 5, stride 2, padding 2, output padding 1 (output 2H x 2W)
 * kind 2 (conv_prepare only): the INPUT-GRADIENT convolution of a stride-1 convolution, prepared straight from that
 *         convolution's weight (Cin, Cout, k, k) = (its Cout, its Cin): flipped taps, swapped channel roles; run with kind 0
 * conv_prepare : weight (Cout, Cin, k, k) [kind 0] / (Cin, Cout, k, k) [kind 1, 2] -> fp16 hi / lo UMMA operand image
 *                (per output channel scaled by a power of two into fp16's normal range; the inverse scales ride along)
 * conv_forward : out = act(conv(x) + bias (+ residual));  x fp32 NCHW with batch stride `x_batch_stride` floats (a
 *                channel slice of a larger tensor is fine), out fp32 NCHW with batch stride `out_batch_stride`,
 *                residual dense (B, Cout, Ho, Wo) or NULL, act: 0 none, 1 GELU (erf), 2 ReLU.
 *                split_hi / split_lo: scratch of conv_split_bytes(B, Cin, H, W) bytes each.
 *                Implicit GEMM on tcgen05, fp16 hi + lo operands in three passes, fp32 accumulation: ~1e-6 relative;
 *                activations beyond +-1.3e5 saturate (fp16 hi + lo range).
 * ------------------------------------------------------------------------------------------------ */
MWA_API int64_t conv_image_bytes(int kind, int Cin, int Cout, int k, int stride);
MWA_API int64_t conv_split_bytes(int B, int Cin, int H, int W);
MWA_API int conv_prepare(const float* w, int kind, int Cin, int Cout, int k, int stride, void* image, int64_t image_bytes,
                         void* stream);
MWA_API int conv_forward(const float* x, int64_t x_batch_stride, const float* bias, const float* residual, float* out,
                         int64_t out_batch_stride, const void* image, void* split_hi, void* split_lo, int kind, int B,
                         int Cin, int Cout, int H, int W, int k, int stride, int act, void* stream);

/* conv_forward_ex : the same kernel with the chaining and epilogue options the transforms use so that an activation
 *   crosses HBM once between two convolutions and the elementwise steps around the slice loop cost no launch:
 *   input   x != NULL: fp32 NCHW as above (in_hi / in_lo are scratch of conv_split_bytes each);
 *           x == NULL: in_hi / in_lo already hold the fp16 hi / lo planes [B][ps*ps][H/ps][W/ps][in_cstride] (ps = 2 for a
 *           stride-2 convolution, else 1) written by a previous call's out_hi / out_lo; the first Cin channels are read
 *           (a channel PREFIX of a wider buffer is a valid input: the reference's torch.cat supports,
 *           models/AutoEncoderRGB_Journal.py:243-259, are prefixes of one buffer);
 *   output  out (fp32 NCHW, may be NULL) and / or out_hi / out_lo: the result as hi / lo planes for the NEXT convolution
 *           (out_ps = that convolution's ps) at channel offset out_coff of a buffer with channel pitch out_cstride
 *           (multiples of 8; channels [Cout, round_up(Cout, 8)) are written as zeros);
 *   act     0 none, 1 GELU, 2 ReLU (after bias + residual), and with v = conv(x) + bias:
 *           3 quantise : out = ste_round(aux - v) + v, out2 (optional) = v      (models/AutoEncoderRGB_Journal.py:257:
 *                        v = mu of the slice, aux = y_slice; bit-identical to quantize_offset_forward on the same v)
 *           4 lrp      : out = aux + 0.5 * tanh(v)                               (:262-264; aux may alias out)
 *           5 gate     : out = aux * sigmoid(v) + residual                       (layers/Masked_Attention.py:186-188:
 *                        v = conv_b's last 1x1, aux = a, residual = x)
 *           6 add2     : out = (v + residual) + aux                              (layers/TransformRGB.py:27, :47: the last
 *                        enhancement block's identity and the DSE skip in one epilogue)
 *           aux: fp32 NCHW (B, Cout, Ho, Wo) with batch stride aux_batch_stride; out2 likewise.
 *   in_scale  NULL, or a DEVICE scalar s (a power of two): the fp32 input is multiplied by s before it is split and the
 *           result divided by s -- for inputs far below fp16's normal range (the gradients of the backward pass). */
/* gemm_tokens_forward : out[t, :] = W x[t, :] + bias for T token rows (token-major, the layout of the attention backward's
 *   scratch tensors) on the convolution kernel: x (T, Cin), out (T, Cout) fp32 row-major, T % 32 == 0, Cout % 8 == 0; `image`
 *   from conv_prepare(k = 1: kind 0 with W (Cout, Cin), or kind 2 with W given as (Cin, Cout)); split_hi / split_lo scratch of
 *   T * round_up(Cin, 8) * 2 bytes each; in_scale as for conv_forward_ex.  Replaces the library GEMMs
 *   qkv = xw Wqkv^T + b, dao = dy Wproj, dxw = dqkv Wqkv of the attention backward. */
MWA_API int gemm_tokens_forward(const float* x, int64_t T, int Cin, const float* bias, float* out, int Cout, const void* image,
                                void* split_hi, void* split_lo, const float* in_scale, void* stream);
/* conv_act_split : fp32 NCHW (B, C, H, W; batch stride x_batch_stride) -> the fp16 hi / lo planes of conv_forward_ex's
 *   x == NULL input, at channel offset out_coff of buffers with channel pitch out_cstride (how an activation that was NOT
 *   produced by one of these convolutions -- GDN, attention, a PixelShuffle -- enters a chain or a support buffer). */
MWA_API int conv_act_split(const float* x, int64_t x_batch_stride, int B, int C, int H, int W, int ps, void* out_hi,
                           void* out_lo, int out_cstride, int out_coff, void* stream);
MWA_API int conv_forward_ex(const float* x, int64_t x_batch_stride, void* in_hi, void* in_lo, int in_cstride,
                            const float* bias, const float* residual, float* out, int64_t out_batch_stride,
                            const float* aux, int64_t aux_batch_stride, float* out2, int64_t out2_batch_stride,
                            void* out_hi, void* out_lo, int out_ps, int out_cstride, int out_coff, const void* image,
                            int kind, int B, int Cin, int Cout, int H, int W, int k, int stride, int act,
                            const float* in_scale, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Masked MS-SSIM (SURVEY.md 8f, rank 4: evaluation on the device)   replaces  metrics/masked_ms_ssim_torch.py:58-121 (_ssim)
 *   and the per-level body of :181-265 (ms_ssim with a mask).
 * ms_ssim_level_forward : X, Y (B, C, H, W) fp32 dense, mask (B, H, W): the mask is binarised (> 0) and multiplied into both
 *     images, the five moments are blurred with the 11-tap Gaussian (sigma 1.5, valid mode, along H then W), and
 *     sums[(b * C + c) * 2 + {0, 1}] receive the SSIM / CS map sums over the positions of the (H-10) x (W-10) valid region
 *     whose nearest-resized mask is non-zero, counts[b] the number of such positions (both overwritten).  H, W >= 11.
 * ms_ssim_pool_forward  : the level's images times the binarised mask, and the binarised mask, through
 *     F.avg_pool2d(2, padding = size % 2): Xo, Yo (B, C, Hp, Wp), Mo (B, Hp, Wp) with Hp = (H + 2 (H % 2) - 2) / 2 + 1.
 * The five-level product (weights 0.0448 ... 0.1333, relu, mean over images and channels) is a handful of scalars. */
MWA_API int ms_ssim_level_forward(const float* X, const float* Y, const float* mask, int B, int C, int H, int W,
                                  float data_range, float* sums, float* counts, void* stream);
MWA_API int ms_ssim_pool_forward(const float* X, const float* Y, const float* mask, int B, int C, int H, int W, float* Xo,
                                 float* Yo, float* Mo, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Range-ANS coder of the bitstream (HOST functions: every pointer is host memory; SURVEY.md 8f, rank 4)   replaces the
 *   compressai.ans calls of models/AutoEncoderRGB_Journal.py:330-368 (BufferedRansEncoder.encode_with_indexes + flush) and
 *   :374-403 (RansDecoder.set_stream + decode_stream): 64-bit rANS state, 32-bit words, 16-bit CDFs chosen per symbol by
 *   `indexes`, 4-bit bypass digits for values outside a CDF's support.  Byte parity with CompressAI is unpinned (absent).
 * cdfs      : (ncdf, cdf_stride) int32; row i has cdf_sizes[i] increasing entries from 0 to 65536; its last interval is the
 *             escape symbol; symbol value = table position + offsets[i]
 * encode    : returns the number of bytes written to `out` (multiple of 4) or a negative MWA_ERR_* (WORKSPACE: too small)
 * decode    : `state` = 4 x int64, zeroed before the first call on a stream; later calls continue where the last stopped */
MWA_API int64_t rans_encode_with_indexes(const int32_t* symbols, const int32_t* indexes, int64_t n, const int32_t* cdfs,
                                         int cdf_stride, const int32_t* cdf_sizes, const int32_t* offsets, int ncdf,
                                         uint8_t* out, int64_t out_capacity);
MWA_API int rans_decode_with_indexes(const uint8_t* stream, int64_t nbytes, int64_t* state, const int32_t* indexes, int64_t n,
                                     const int32_t* cdfs, int cdf_stride, const int32_t* cdf_sizes, const int32_t* offsets,
                                     int ncdf, int32_t* symbols_out);

/* ------------------------------------------------------------------------------------------------
 * Lane-interleaved rANS on the device (csrc/rans_dev.cu; DESIGN.md 4.7)   the same coder as above, on the GPU, for a stream
 *   format whose message is split across L lanes: element g of a stream (counted across all decode calls) belongs to lane
 *   g mod L, and lane l's segment is byte for byte what rans_encode_with_indexes writes for elements l, l + L, l + 2L, ...
 *   Stream layout, little-endian u32 words:
 *     MWA_RANS_LANES_MAGIC, 0x80000000 | MWA_RANS_LANES_VERSION, L, L lane byte lengths (multiples of 4, >= 8), segments.
 *   Word 1 has its top bit set; in a host-format stream word 1 is the high half of a final state in [2^31, 2^63), so < 2^31.
 *   Device pointers, asynchronous on `stream`; tables as for the host coder (cdfs / cdf_sizes / offsets, device copies).
 * rans_lanes_encode : symbols, indexes (n_streams, n) int32.  Thread (s, l) writes lane l of stream s into slot s * lanes + l
 *             of `slots` (n_streams * lanes slots of slot_words u32 each; the segment ends at the slot's end) and sets
 *             lane_words[s * lanes + l] to its length in words, or MWA_ERR_WORKSPACE when the slot is too small (nothing is
 *             written past it: retry with larger slots), or MWA_ERR_INVALID for an index outside [0, ncdf) / a broken row.
 * rans_lanes_pack   : after rans_lanes_encode on the same slots: writes every stream, header included, back to back into
 *             `out` (out_words u32; n_streams * (3 + lanes + lanes * slot_words) always suffice), stream_bytes[s] = byte
 *             length of stream s and stream_bytes[n_streams] = total bytes, or the negative status of a failed lane
 *             (INVALID before WORKSPACE), in which case `out` holds no streams.  lane_dst: n_streams * lanes int64 scratch.
 * rans_lanes_decode : data = the streams of the call (data_words u32); lane_state (total_lanes, 4) int64, one row per lane of
 *             every stream: {x, next word, end word, stream + 2^32 lane}, prepared by the caller as {0, index of the lane
 *             segment's first word in data, one past its last, ...} and updated by each call, so successive calls continue
 *             each stream; stream_lanes[s] = L of stream s (streams may differ).  Decodes elements [position, position + n)
 *             of every stream with indexes (n_streams, n) into symbols (n_streams, n).  A truncated or corrupt segment or
 *             an index outside [0, ncdf) sets status[s] (int32, zeroed by the caller) to MWA_ERR_INVALID; that stream's
 *             later lanes and calls stop, its symbols are then undefined.  The return value covers the arguments only. */
#define MWA_RANS_LANES_MAGIC 0x4C41574Du   /* "MWAL" */
#define MWA_RANS_LANES_VERSION 1u
MWA_API int rans_lanes_encode(const int32_t* symbols, const int32_t* indexes, int n_streams, int64_t n, int lanes,
                              const int32_t* cdfs, int cdf_stride, const int32_t* cdf_sizes, const int32_t* offsets,
                              int ncdf, uint32_t* slots, int64_t slot_words, int32_t* lane_words, void* stream);
MWA_API int rans_lanes_pack(const uint32_t* slots, int64_t slot_words, const int32_t* lane_words, int n_streams, int lanes,
                            int64_t* lane_dst, int64_t* stream_bytes, uint32_t* out, int64_t out_words, void* stream);
MWA_API int rans_lanes_decode(const uint32_t* data, int64_t data_words, int64_t* lane_state, int total_lanes,
                              const int32_t* stream_lanes, int n_streams, const int32_t* indexes, int64_t n,
                              int64_t position, const int32_t* cdfs, int cdf_stride, const int32_t* cdf_sizes,
                              const int32_t* offsets, int ncdf, int32_t* symbols, int32_t* status, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Rate / distortion terms of the forward (csrc/rate.cu)   replaces  models/AutoEncoderRGB_Journal.py:36-64 (reconstruct_error)
 * and :283-291 (bits of y under the Gaussian conditional, of z under the factorised prior, bpp), which the reference runs
 * as ~90 elementwise / reduction / batched-GEMM launches: one pass per term + a finalize launch, inference only.
 *   input, x_hat (B, C, H, W), mask (B, 1, H, W): squared error over the pixels with mask > 0, per image / (C * count), mean;
 *   y, scales, means: n_y elements each;   z_hat (B, Cz, hw_z) with eb_params = HOST array of 14 device pointers
 *   [_matrix0.._matrix4, _bias0.._bias4, _factor0.._factor3] of the factorised prior with filters (3, 3, 3, 3);
 *   out4 (device) = [mse, y bpp, z bpp, y bpp + z bpp], bpp = bits / (B * H * W).  workspace: rate_workspace_bytes(B), 8-aligned.
 * ------------------------------------------------------------------------------------------------ */
MWA_API int64_t rate_workspace_bytes(int B);
MWA_API int rate_forward(const float* input, const float* x_hat, const float* mask, int B, int C, int H, int W, const float* y,
                 const float* scales, const float* means, int64_t n_y, const float* z_hat, const float* const* eb_params,
                 int Cz, int64_t hw_z, void* workspace, int64_t workspace_bytes, float* out4, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MWA_B200_H_ */
