"""The reference's OWN model files import and build on top of the drop-in modules (only where MWA_REFERENCE_ROOT names
the original project's tree; runs in a subprocess because it re-binds the top-level `layers` package)."""
import os
import subprocess
import sys

import pytest

from oracle import live_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r"""
import sys, os, torch
sys.path.insert(0, %(root)r)
sys.dont_write_bytecode = True
import mwa_b200
mwa_b200.install(%(ref)r, extra_paths=[os.path.join(%(root)r, "oracle", "shims")])
from models.AutoEncoderRGB_Journal import AutoEncoder
import models.AutoEncoderRGB_Journal as rgb_mod
from models.AutoEncoderMask_Journal import AutoEncoder as MaskAutoEncoder
import layers.GDN, layers.masked_win_attention
assert layers.GDN.GDN is mwa_b200.GDN
torch.manual_seed(234)
net, masknet = AutoEncoder(), MaskAutoEncoder()
mods = [type(m) for m in net.modules()]
assert mods.count(mwa_b200.GDN) == 6, mods.count(mwa_b200.GDN)
assert mods.count(mwa_b200.MaskedWinBasedAttention) == 4
assert [type(m) for m in masknet.modules()].count(mwa_b200.GDN) == 6
mwa_b200.patch_model_rounding(rgb_mod)
assert rgb_mod.ste_round is mwa_b200.ste_round
keys = sorted(net.state_dict().keys())
print("KEYS", len(keys), sum(p.numel() for p in net.parameters()))
for k in keys: print(k)
"""

REF_SCRIPT = r"""
import sys, os, torch
sys.dont_write_bytecode = True
sys.path.insert(0, os.path.join(%(root)r, "oracle", "shims")); sys.path.insert(0, %(ref)r)
from models.AutoEncoderRGB_Journal import AutoEncoder
torch.manual_seed(234)
net = AutoEncoder()
keys = sorted(net.state_dict().keys())
print("KEYS", len(keys), sum(p.numel() for p in net.parameters()))
for k in keys: print(k)
"""


@pytest.mark.skipif(not live_reference.available(), reason="needs MWA_REFERENCE_ROOT: the original project's source tree")
def test_reference_models_build_on_dropins_with_identical_checkpoint_keys():
    fmt = dict(root=ROOT, ref=live_reference.REFERENCE_ROOT)
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    ours = subprocess.run([sys.executable, "-c", SCRIPT % fmt], capture_output=True, text=True, env=env, timeout=600)
    assert ours.returncode == 0, ours.stderr[-3000:]
    theirs = subprocess.run([sys.executable, "-c", REF_SCRIPT % fmt], capture_output=True, text=True, env=env,
                            timeout=600)
    assert theirs.returncode == 0, theirs.stderr[-3000:]
    assert ours.stdout == theirs.stdout          # same key list, same parameter count
    assert "Encoder.attention1.attn.attn.qkv.weight" in ours.stdout
    assert "Encoder.gdn1.gamma" in ours.stdout
