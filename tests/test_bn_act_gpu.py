"""GPU parity of the fused BatchNorm + LeakyReLU + Dropout kernels (channels-last bf16) against
torch's batch_norm / leaky_relu on the same bf16 input, forward, backward and running statistics."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("B,C,H,W", [(4, 16, 64, 64), (2, 32, 32, 32), (2, 64, 16, 16), (2, 128, 8, 8), (2, 256, 16, 16),
                                     (1, 16, 48, 40)])
def test_bn_lrelu_matches_torch(B, C, H, W):
    from uaps_b200.bn_act import bn_lrelu_dropout
    dev = torch.device("cuda:0")
    g = torch.Generator().manual_seed(C + H)
    y = (torch.randn(B, C, H, W, generator=g) * 1.7 + 0.3).to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    bn_a, bn_b = torch.nn.BatchNorm2d(C).to(dev), torch.nn.BatchNorm2d(C).to(dev)
    with torch.no_grad():
        bn_a.weight.copy_(1 + 0.2 * torch.randn(C, generator=g)); bn_a.bias.copy_(0.2 * torch.randn(C, generator=g))
        bn_b.load_state_dict(bn_a.state_dict())
    cot = torch.randn(B, C, H, W, generator=g).to(dev)
    # reference in fp32 on the bf16-rounded input
    yr = y.float().requires_grad_(True)
    ref = F.leaky_relu(bn_a(yr), 0.01)
    (ref * cot).sum().backward()
    yo = y.clone().requires_grad_(True)
    out = bn_lrelu_dropout(yo, bn_b, 0.0)
    (out.float() * cot).sum().backward()
    assert out.dtype == torch.bfloat16 and out.is_contiguous(memory_format=torch.channels_last)
    assert (out.float() - ref).abs().max().item() <= 1e-2 * ref.abs().max().item()
    gscale = yr.grad.abs().max().item()
    assert (yo.grad.float() - yr.grad).abs().max().item() <= 2e-2 * gscale
    assert torch.allclose(bn_b.weight.grad, bn_a.weight.grad, rtol=2e-2, atol=2e-2 * bn_a.weight.grad.abs().max().item())
    assert torch.allclose(bn_b.bias.grad, bn_a.bias.grad, rtol=2e-2, atol=2e-2 * bn_a.bias.grad.abs().max().item())
    assert torch.allclose(bn_b.running_mean, bn_a.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(bn_b.running_var, bn_a.running_var, rtol=1e-4, atol=1e-5)
    assert int(bn_b.num_batches_tracked) == 1


def test_fused_dropout_is_consistent_between_forward_and_backward():
    from oracle.philox_ref import bn_keep, keep_scale
    from uaps_b200.bn_act import bn_lrelu_dropout
    dev = torch.device("cuda:0")
    C = 32
    y = torch.randn(4, C, 32, 32, device=dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    bn = torch.nn.BatchNorm2d(C).to(dev)
    for p in (0.05, 0.3, 0.5):
        yo = y.clone().requires_grad_(True)
        out = bn_lrelu_dropout(yo, bn, p, seed=7)
        base = bn_lrelu_dropout(y, bn, 0.0)
        kept = out != 0
        assert kept.float().mean().item() == pytest.approx(1 - p, abs=0.02)
        scale = 1.0 / (1.0 - p)
        assert torch.allclose(out.float()[kept], (base.float() * scale)[kept], rtol=2e-2, atol=1e-3)
        # same seed -> same mask
        assert torch.equal(bn_lrelu_dropout(y, bn, p, seed=7) != 0, kept)
        # the mask is Philox(seed 7, stream 21) of the chunk index, bit for bit (oracle/philox_ref.py)
        want = torch.from_numpy(bn_keep(7, y.numel() // C, C, p)).to(dev)
        rows = lambda t: t.permute(0, 2, 3, 1).reshape(-1, C)
        nz = rows(base) != 0
        assert torch.equal(rows(kept)[nz], want[nz])
        # backward regenerates it: d beta = sum(g * keep * keep_scale * leaky_relu'(z)) over the oracle's mask
        bn.weight.grad = bn.bias.grad = None
        out.float().sum().backward()
        assert torch.isfinite(yo.grad.float()).all()
        d = torch.where(rows(base) > 0, 1.0, 0.01).double() * want.double() * float(keep_scale(p))
        assert torch.allclose(bn.bias.grad.double(), d.sum(0), rtol=1e-5, atol=1e-3)
