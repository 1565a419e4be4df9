"""Oracle restatement vs the LIVE reference modules (only where MWA_REFERENCE_ROOT names the original project's tree)."""
import pytest
import torch

from oracle import live_reference
from oracle import ref_ops as R

pytestmark = pytest.mark.skipif(not live_reference.available(), reason="needs MWA_REFERENCE_ROOT: the original project's source tree")


@pytest.fixture(scope="module")
def ref():
    return live_reference.load()


@pytest.mark.parametrize("C,heads,ws,s,B,H,W", [(192, 8, 8, 4, 1, 16, 24), (80, 8, 4, 2, 2, 8, 12),
                                                (192, 6, 8, 0, 1, 16, 16), (24, 2, 2, 1, 3, 4, 6)])
def test_masked_and_unmasked_blocks(ref, C, heads, ws, s, B, H, W):
    torch.manual_seed(C + ws + s)
    m = ref.masked.WinBasedAttention(dim=C, num_heads=heads, window_size=ws, shift_size=s)
    u = ref.unmasked.WinBasedAttention(dim=C, num_heads=heads, window_size=ws, shift_size=s)
    with torch.no_grad():
        m.attn.relative_position_bias_table.normal_(0, 0.5)
    u.load_state_dict(m.state_dict())
    x = torch.randn(B, C, H, W)
    alpha = (torch.rand(B, 1, H // ws, W // ws) > 0.4).float().repeat_interleave(ws, 2).repeat_interleave(ws, 3)
    alpha = torch.roll(alpha * torch.rand(B, 1, H, W), (s, s), (2, 3))
    a = m.attn
    args = (a.qkv.weight, a.qkv.bias, a.proj.weight, a.proj.bias, a.relative_position_bias_table, heads, ws, s)
    with torch.no_grad():
        assert torch.equal(m(x, alpha), R.masked_window_attention(x, alpha, *args))
        assert torch.equal(u(x), R.masked_window_attention(x, None, *args))
        # property 1 (SURVEY.md section 4): alpha == 1 everywhere -> masked == unmasked, bit exact
        assert torch.equal(m(x, torch.ones(B, 1, H, W)), u(x))
        keep = R.window_keep(alpha, ws, s)
        assert torch.equal(keep, ref.masked.remove_zero_windows(
            ref.masked.window_partition(torch.roll(x.permute(0, 2, 3, 1), (-s, -s), (1, 2)), ws),
            ref.masked.window_partition(torch.roll(alpha.permute(0, 2, 3, 1), (-s, -s), (1, 2)), ws))[1])


def test_window_attention_tokens_with_mask(ref):
    torch.manual_seed(5)
    wa = ref.masked.WindowAttention(dim=32, window_size=(4, 4), num_heads=4)
    x = torch.randn(6, 16, 32)
    mask = torch.randn(3, 16, 16)
    with torch.no_grad():
        y = wa(x, mask)
        y2 = R.window_attention(x, wa.qkv.weight, wa.qkv.bias, wa.proj.weight, wa.proj.bias,
                                wa.relative_position_bias_table, 4, 4, mask=mask.repeat(2, 1, 1))
    torch.testing.assert_close(y, y2, rtol=1e-5, atol=1e-6)
    assert torch.equal(wa.relative_position_index, R.relative_position_index(4))


@pytest.mark.parametrize("inverse", [False, True])
def test_gdn(ref, inverse):
    torch.manual_seed(9)
    g = ref.gdn.GDN(48, inverse=inverse)
    with torch.no_grad():
        g.gamma.add_(torch.rand(48, 48) * 0.05)
        g.beta.mul_(torch.rand(48) + 0.5)
        g.beta[::5] = 1e-6
    x = (torch.randn(2, 48, 6, 10) * 3).requires_grad_(True)
    y = g(x)
    y.sum().backward()
    x2 = x.detach().clone().requires_grad_(True)
    b2 = g.beta.detach().clone().requires_grad_(True)
    g2 = g.gamma.detach().clone().requires_grad_(True)
    y2 = R.gdn(x2, b2, g2, inverse=inverse)
    y2.sum().backward()
    torch.testing.assert_close(y, y2, rtol=2e-5, atol=2e-6)
    torch.testing.assert_close(x.grad, x2.grad, rtol=1e-4, atol=1e-5)
    torch.testing.assert_close(g.beta.grad, b2.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(g.gamma.grad, g2.grad, rtol=1e-4, atol=1e-4)
    pedestal, bb, gb = R.gdn_constants()
    assert (pedestal, bb, gb) == (g.pedestal, g.beta_bound, g.gamma_bound)


def test_alpha_pyramid_matches_supplymask(ref):
    import importlib
    sm = importlib.import_module("layers.SupplyMask").SupplyMaskToTransform()
    a = torch.rand(1, 1, 64, 96)
    for mine, theirs in zip(R.alpha_pyramid(a), sm(a)):
        assert torch.equal(mine, theirs)
