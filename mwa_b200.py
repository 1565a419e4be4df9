"""Import alias: the package directory name required by the build contains hyphens
(`deep-learning-based-rgba-image-compression-with-masked-window-based-attention_b200`), which the
`import` statement cannot spell.  `import mwa_b200` loads it and re-exports its public pieces.
"""
import importlib
import os
import sys

PACKAGE_NAME = "deep-learning-based-rgba-image-compression-with-masked-window-based-attention_b200"
_root = os.path.dirname(os.path.abspath(__file__))
if _root not in sys.path:
    sys.path.insert(0, _root)

package = importlib.import_module(PACKAGE_NAME)
_abi = importlib.import_module(PACKAGE_NAME + "._abi")
build_mod = importlib.import_module(PACKAGE_NAME + ".build")
quant = importlib.import_module(PACKAGE_NAME + ".quant")
_install = importlib.import_module(PACKAGE_NAME + ".install")
GDN_mod = importlib.import_module(PACKAGE_NAME + ".layers.GDN")
masked_win_attention = importlib.import_module(PACKAGE_NAME + ".layers.masked_win_attention")
win_attention = importlib.import_module(PACKAGE_NAME + ".layers.win_attention")
Masked_Attention = importlib.import_module(PACKAGE_NAME + ".layers.Masked_Attention")
SupplyMask = importlib.import_module(PACKAGE_NAME + ".layers.SupplyMask")
data_parallel = importlib.import_module(PACKAGE_NAME + ".data_parallel")
conv = importlib.import_module(PACKAGE_NAME + ".layers.conv")
codec = importlib.import_module(PACKAGE_NAME + ".codec")
metrics = importlib.import_module(PACKAGE_NAME + ".metrics")
pipeline = importlib.import_module(PACKAGE_NAME + ".pipeline")
_params = importlib.import_module(PACKAGE_NAME + ".layers._params")
rgba8 = importlib.import_module(PACKAGE_NAME + ".rgba8")

GDN = GDN_mod.GDN
LowerBound = GDN_mod.LowerBound
MaskedWinBasedAttention = masked_win_attention.WinBasedAttention
WinBasedAttention = win_attention.WinBasedAttention
WindowAttention = masked_win_attention.WindowAttention
Win_noShift_Attention = Masked_Attention.Win_noShift_Attention
gate_residual = Masked_Attention.gate_residual
SupplyMaskToTransform = SupplyMask.SupplyMaskToTransform
alpha_pyramid = SupplyMask.alpha_pyramid
constraint = SupplyMask.constraint
ste_round = quant.ste_round
quantize_offset = quant.quantize_offset
lrp_add = quant.lrp_add
quantize_levels = quant.quantize_levels
install = _install.install
patch_model_rounding = _install.patch_model_rounding
accelerate_convs = _install.accelerate_convs
uninstall = _install.uninstall
build = build_mod.build
GradientAllReduce = data_parallel.GradientAllReduce
RGBACodec = codec.AutoEncoder
masked_ms_ssim = metrics.masked_ms_ssim
masked_psnr = metrics.masked_psnr
HostPipeline = pipeline.HostPipeline
invalidate_param_blocks = _params.invalidate_param_blocks
rgba8_ingest = rgba8.rgba8_ingest
rgba8_egress = rgba8.rgba8_egress
rgba16_ingest = rgba8.rgba16_ingest
rgba16_egress = rgba8.rgba16_egress
tile_grid = rgba8.tile_grid
ingest_tiles = rgba8.ingest_tiles
egress_tiles = rgba8.egress_tiles
MwaB200Error = _abi.MwaB200Error
ALGO_AUTO, ALGO_SIMT, ALGO_TCGEN05 = _abi.ALGO_AUTO, _abi.ALGO_SIMT, _abi.ALGO_TCGEN05
