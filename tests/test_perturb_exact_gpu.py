"""The Philox perturbation kernels bit for bit against the host oracle (oracle/philox_ref.py): the channels-last bf16
perturb3_nhwc (FeatureNoise shared by the batch across its groups of 8 samples, Dropout per element, device-resident key
and threshold) and the fp32 NCHW perturb3 / FeatureNoise / Dropout at both vector widths."""
import numpy as np
import pytest
import torch

from oracle import philox_ref as R

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
U = 2.0 ** -24


def _bf16_ulp(x):
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), e - 8)


def _to_bf16(x64):
    """fp64 -> fp32 (one rounding, as the kernel's fp32 result) -> bf16 (round to nearest even, as its store)."""
    return x64.float().to(torch.bfloat16)


def _rows(t):
    """[B,C,H,W] channels-last -> [B, HW, C] in memory order."""
    return t.permute(0, 2, 3, 1).reshape(t.shape[0], -1, t.shape[1])


def _x_nhwc(B, C, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, C, H, W, generator=g) * 2).to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)


@pytest.mark.parametrize("B", [1, 7, 9, 17, 64])
@pytest.mark.parametrize("C,p", [(16, 0.5), (32, 0.3)])
def test_perturb3_nhwc_matches_oracle_bit_for_bit(B, C, p):
    from uaps_b200.perturb import perturb3_nhwc
    H, W, seed, rng = 8, 12, 0xABCDEF + B, 0.3
    x = _x_nhwc(B, C, H, W, B + C)
    yn, yd, _ = perturb3_nhwc(x, seed=seed, u=0.8, p=p, uniform_range=rng)
    X = _rows(x).double()
    n = torch.from_numpy(R.nhwc_noise(seed, H * W, C, rng)).double().to(DEV)          # one draw for every sample
    keep = torch.from_numpy(R.nhwc_keep(seed, B, H * W, C, p)).to(DEV)
    assert torch.equal(_rows(yn), _to_bf16(X * n + X))                                 # fmaf(v, n, v): exact in fp64
    scale = float(R.keep_scale(p))
    assert torch.equal(_rows(yd), _to_bf16(torch.where(keep, X * scale, torch.zeros_like(X))))


@pytest.mark.parametrize("aliases", [0, 2])
@pytest.mark.parametrize("B", [7, 17])
def test_perturb3_nhwc_backward_within_one_ulp(B, aliases):
    from uaps_b200.perturb import perturb3_nhwc
    C, H, W, seed, p, rng = 16, 8, 6, 99 + B, 0.5, 0.3
    x = _x_nhwc(B, C, H, W, 3 * B).requires_grad_(True)
    outs = perturb3_nhwc(x, seed=seed, u=0.8, p=p, uniform_range=rng, outputs=(True, True, False), aliases=aliases)
    assert outs[2] is None
    live = [o for o in outs if o is not None]
    cots = [_x_nhwc(B, C, H, W, 1000 + i) for i in range(len(live))]
    torch.autograd.backward(live, cots)
    n = torch.from_numpy(R.nhwc_noise(seed, H * W, C, rng)).double().to(DEV)
    keep = torch.from_numpy(R.nhwc_keep(seed, B, H * W, C, p)).to(DEV).double() * float(R.keep_scale(p))
    G = [_rows(c).double() for c in cots]
    terms = [G[0] * n + G[0], G[1] * keep] + G[2:]
    want = sum(terms)
    mag = sum(t.abs() for t in terms)
    err = (_rows(x.grad).double() - want).abs()
    assert (err <= _bf16_ulp(want) + 8 * U * mag).all()


def test_perturb3_nhwc_device_key_and_threshold():
    """seed_dev: the kernel adds the uint64 at that address to ``seed`` (mod 2^64); u_dev replaces u."""
    from uaps_b200.perturb import perturb3_nhwc
    B, C, H, W, seed = 9, 16, 4, 8, (1 << 64) - 7
    x = _x_nhwc(B, C, H, W, 5)
    key_val = 0x0123_4567_89AB_CDEF
    key = torch.tensor([key_val], dtype=torch.int64, device=DEV)
    uval = torch.tensor([0.75], dtype=torch.float32, device=DEV)
    yn, yd, yf = perturb3_nhwc(x, seed=seed, u=0.9, seed_dev=key.data_ptr(), u_dev=uval.data_ptr())
    eff = (seed + key_val) & R.MASK64
    rn, rd, rf = perturb3_nhwc(x, seed=eff, u=0.75)
    assert torch.equal(yn, rn) and torch.equal(yd, rd) and torch.equal(yf, rf)
    X = _rows(x).double()
    n = torch.from_numpy(R.nhwc_noise(eff, H * W, C, 0.3)).double().to(DEV)
    assert torch.equal(_rows(yn), _to_bf16(X * n + X))
    keep = torch.from_numpy(R.nhwc_keep(eff, B, H * W, C, 0.5)).to(DEV)
    assert torch.equal(_rows(yd) != 0, keep & (X != 0))
    # and the backward regenerates the same draw from the device key
    xg = x.clone().requires_grad_(True)
    outs = perturb3_nhwc(xg, seed=seed, u=0.9, seed_dev=key.data_ptr(), u_dev=uval.data_ptr(), outputs=(False, True, False))
    outs[1].backward(torch.ones_like(x))
    assert torch.equal(_rows(xg.grad).float(), keep.float() * float(R.keep_scale(0.5)))


# fp32 NCHW: HW % 4 == 0 selects the 4-wide kernels of perturb3, HW % 4 != 0 the scalar ones; chw (FeatureNoise) and
# n (Dropout) select theirs the same way
@pytest.mark.parametrize("shape", [(2, 3, 8, 12), (3, 5, 5, 7), (2, 4, 3, 3), (1, 2, 9, 6)])
def test_perturb3_fp32_matches_oracle_bit_for_bit(shape):
    from uaps_b200 import perturb as P
    B, C, H, W = shape
    seed, p, rng = 0x1234_5678_9ABC + B * C, 0.5, 0.3
    g = torch.Generator().manual_seed(sum(shape))
    x = (torch.randn(shape, generator=g) * 2).to(DEV)
    yn, yd, _ = P.perturb3(x, seed=seed, u=0.8, p=p, uniform_range=rng)
    xs = x.cpu().numpy().reshape(B, -1)
    n = R.nchw_noise(seed, C * H * W, rng)
    want_n = (xs * n) + xs                                   # float32 arithmetic: __fmul_rn then __fadd_rn
    assert want_n.dtype == np.float32
    assert np.array_equal(yn.cpu().numpy().reshape(B, -1), want_n)
    keep = R.nchw_keep(seed, xs.size, p).reshape(B, -1)
    want_d = (xs * keep.astype(np.float32)) * R.keep_scale(p)
    assert np.array_equal(yd.cpu().numpy().reshape(B, -1), want_d)
    # the stand-alone kernels draw the same streams
    assert np.array_equal(P.FeatureNoise(rng)(x, seed=seed).cpu().numpy().reshape(B, -1), want_n)
    assert np.array_equal(P.Dropout(x, p, seed=seed).cpu().numpy().reshape(B, -1), want_d)
