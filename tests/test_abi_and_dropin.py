"""CPU-side checks of the boundary: the C ABI exports what include/mwa_b200.h declares, argument validation
that happens before any CUDA call, and the drop-in nn.Module surface (signatures, state-dict keys)."""
import ctypes
import inspect
import os
import re

import pytest
import torch

from oracle import live_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "mwa_b200.h")).read()
    return re.findall(r"MWA_API\s+[\w\s\*]+?\b(\w+)\s*\(", text)


def test_library_exports_every_declared_symbol(pkg):
    lib = ctypes.CDLL(pkg._abi.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/mwa_b200.h but not exported"
    assert set(declared) == set(pkg._abi.EXPORTED_SYMBOLS), "ctypes binding and header drifted apart"


def test_library_has_no_torch_dependency(pkg):
    import subprocess
    out = subprocess.run(["ldd", pkg._abi.LIB_PATH], capture_output=True, text=True).stdout
    # dependency names and paths only: the load addresses ldd prints are random hex that may contain "c10"
    deps = " ".join(tok for line in out.splitlines() for tok in line.split() if not tok.startswith("(0x"))
    assert deps.strip()
    assert "torch" not in deps and "c10" not in deps and "libcudart" not in deps   # cudart linked statically


def test_status_strings_and_sizes(lib):
    assert lib.mwa_b200_abi_version() == 1
    assert lib.mwa_b200_status_string(0) == b"ok"
    assert b"invalid" in lib.mwa_b200_status_string(-1)
    assert lib.gdn_param_bytes(192) > 2 * 4 * 192 * 192
    assert lib.gdn_param_bytes(0) < 0
    assert lib.mwa_param_bytes(192, 8, 8) > 4 * 4 * 192 * 192
    assert lib.mwa_param_bytes(192, 7, 8) < 0                 # C % heads != 0
    assert lib.gdn_backward_workspace_bytes(2, 192, 64) >= 4 * 2 * 192 * 64


def test_argument_validation_without_gpu(lib):
    """these return before touching the device"""
    one = ctypes.c_void_p(16)
    assert lib.mwa_forward(None, None, None, None, 1, 192, 8, 8, 8, 8, 0, 0, 0, None, None, 0, None) == -1
    assert lib.mwa_forward(one, None, one, one, 1, 192, 8, 8, 8, 8, 8, 0, 0, None, None, 0, None) == -1     # shift >= ws
    assert lib.mwa_forward(one, None, one, one, 1, 192, 12, 8, 8, 8, 0, 0, 0, None, None, 0, None) == -1    # H % ws
    for algo in (3, 4, 5):                                                                          # unknown algo
        assert lib.mwa_forward(None, None, None, None, 0, 192, 8, 8, 8, 8, 0, 0, algo, None, None, 0, None) == -1
    assert lib.mwa_workspace_bytes(16, 128, 192, 8) >= 5 * 6144
    assert lib.gdn_forward(None, None, None, 1, 192, 64, 0, 0, 0, None) == -1
    assert lib.gdn_forward(one, one, one, 0, 192, 64, 0, 0, 0, None) == 0                          # empty batch
    assert lib.round_ste_forward(one, one, 0, 0, 0, 0, None) == 0                                  # empty input
    assert lib.round_ste_forward(None, one, 1, 4, 4, 4, None) == -1
    assert lib.quantize_levels_forward(one, one, 4, 0.0, None) == -1


def test_cpu_tensors_fail_loudly(pkg):
    g = pkg.GDN(8)
    with pytest.raises(pkg.MwaB200Error, match="no CPU fallback"):
        g(torch.randn(1, 8, 4, 4))
    a = pkg.MaskedWinBasedAttention(16, 2, 4, 2)
    with pytest.raises(pkg.MwaB200Error):
        a(torch.randn(1, 16, 8, 8), torch.ones(1, 1, 8, 8))
    with pytest.raises(pkg.MwaB200Error):
        pkg.ste_round(torch.randn(4))


def test_constructor_contracts(pkg):
    with pytest.raises(AssertionError):
        pkg.MaskedWinBasedAttention(192, 8, 8, 8)             # shift_size must be < window_size
    with pytest.raises(NotImplementedError):
        pkg.MaskedWinBasedAttention(192, 8, 8, 0, drop_path=0.1)
    a = pkg.MaskedWinBasedAttention()
    assert (a.dim, a.num_heads, a.window_size, a.shift_size) == (192, 8, 8, 0)
    assert sorted(a.state_dict()) == ["attn.proj.bias", "attn.proj.weight", "attn.qkv.bias", "attn.qkv.weight",
                                      "attn.relative_position_bias_table", "attn.relative_position_index"]
    assert a.attn.relative_position_index.dtype == torch.int64
    assert a.attn.relative_position_bias_table.shape == (225, 8)
    g = pkg.GDN(192, inverse=True)
    assert sorted(g.state_dict()) == ["beta", "gamma"]
    assert g.pedestal == 2 ** -36 and g.gamma_bound == 2 ** -18
    # effective beta = 1, gamma = 0.1 * I at init (SURVEY.md 3.4)
    torch.testing.assert_close(g.beta ** 2 - g.pedestal, torch.ones(192))
    torch.testing.assert_close(g.gamma ** 2 - g.pedestal, 0.1 * torch.eye(192), atol=1e-7, rtol=0)


@pytest.mark.skipif(not live_reference.available(), reason="needs MWA_REFERENCE_ROOT: the original project's source tree")
class TestAgainstReferenceSurface:
    def test_signatures_match(self, pkg):
        ref = live_reference.load()
        pairs = [(ref.masked.WinBasedAttention, pkg.masked_win_attention.WinBasedAttention),
                 (ref.masked.WindowAttention, pkg.masked_win_attention.WindowAttention),
                 (ref.unmasked.WinBasedAttention, pkg.win_attention.WinBasedAttention),
                 (ref.gdn.GDN, pkg.GDN_mod.GDN)]
        for theirs, ours in pairs:
            assert str(inspect.signature(theirs.__init__)) == str(inspect.signature(ours.__init__)), theirs
            assert list(inspect.signature(theirs.forward).parameters) == \
                list(inspect.signature(ours.forward).parameters), theirs
        for name in ("window_partition", "window_reverse", "remove_zero_windows", "WindowAttention",
                     "WinBasedAttention", "torch", "nn"):
            assert hasattr(pkg.masked_win_attention, name)
        for name in ("LowerBound", "GDN", "torch", "nn", "F", "optim", "Function"):
            assert hasattr(pkg.GDN_mod, name)

    def test_state_dict_round_trip(self, pkg):
        ref = live_reference.load()
        for kw in (dict(dim=192, num_heads=8, window_size=8, shift_size=4),
                   dict(dim=80, num_heads=8, window_size=4, shift_size=2)):
            theirs = ref.masked.WinBasedAttention(**kw)
            ours = pkg.masked_win_attention.WinBasedAttention(**kw)
            ours.load_state_dict(theirs.state_dict(), strict=True)
            theirs.load_state_dict(ours.state_dict(), strict=True)
            assert torch.equal(ours.attn.relative_position_index, theirs.attn.relative_position_index)
        theirs, ours = ref.gdn.GDN(192), pkg.GDN(192)
        assert torch.equal(theirs.beta, ours.beta) and torch.equal(theirs.gamma, ours.gamma)
        ours.load_state_dict(theirs.state_dict(), strict=True)

    def test_helper_functions_match(self, pkg):
        ref = live_reference.load()
        x = torch.randn(2, 16, 24, 5)
        assert torch.equal(ref.masked.window_partition(x, 8), pkg.masked_win_attention.window_partition(x, 8))
        w = ref.masked.window_partition(x, 8)
        assert torch.equal(ref.masked.window_reverse(w, 8, 16, 24), pkg.masked_win_attention.window_reverse(w, 8, 16, 24))
        a = (torch.rand(w.shape[0], 8, 8, 1) > 0.5).float() * (torch.rand(w.shape[0], 1, 1, 1) > 0.5)
        r1, m1 = ref.masked.remove_zero_windows(w, a)
        r2, m2 = pkg.masked_win_attention.remove_zero_windows(w, a)
        assert torch.equal(r1, r2) and torch.equal(m1, m2)
        v = torch.tensor([0.5, 2.0], requires_grad=True)
        v2 = v.detach().clone().requires_grad_(True)
        ref.gdn.LowerBound.apply(v, 1.0).sum().backward()
        pkg.LowerBound.apply(v2, 1.0).sum().backward()
        assert torch.equal(v.grad, v2.grad)
