"""Fused BatchNorm + LeakyReLU + Dropout (channels-last bf16) element by element against an fp64 reference that uses the
host-regenerated Philox mask (oracle/philox_ref.py), forward, backward and running statistics, on every path training
takes: the statistics pass, replicated sums, the conv epilogue's sums, the device-resident step and the encoder block.

Error bounds.  u = 2^-24 (fp32 unit roundoff).  The kernel forms, per channel, mean and var in fp64 from fp32-accumulated
sums, rstd = fl32(1 / sqrt(var + eps)), sc = fl32(gamma * rstd), sh = fl32(beta - mean * sc) and per element
z = fl32(y * sc + sh), then LeakyReLU, the keep mask and keep_scale in fp32, and one rounding to bf16.  Against
z_ref = gamma * rstd_ref * (y - mean_ref) + beta in fp64:

  |z - z_ref| <= Ez = |gamma| rstd (|y - mean| * rel_rstd + dmean) + 8u (|y gamma rstd| + |mean gamma rstd| + |beta|)

where the last term covers the four fp32 roundings of sc, sh and z (8u for two each), and dmean / rel_rstd are the
statistics' errors: an fp32 sum whose longest chain of additions is K has error <= K u sum|term| (K = grid-stride loop
trips + 5 warp shuffles + 8 shared-memory adds + slack), and a channel whose values are multiples of q with
sum|y| < 2^24 q (and sum y^2 < 2^24 q^2) is summed exactly.  The bf16 output is then within one bf16 ulp of the
reference plus the propagated Ez; dropped elements are exactly 0.  Elements with |z_ref| <= Ez may take either
LeakyReLU branch: they are left out of the elementwise checks, their possible gradient flip (1 - slope)|g| is added to
the bounds of the per-channel gradient sums, and the tests assert that they are rare.  The gradient bounds follow the
same way from the backward kernels' arithmetic (see ``_bounds``).
"""
import numpy as np
import pytest
import torch

from oracle import philox_ref as R

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
SLOPE = float(np.float32(0.01))          # the kernel's fp32 slope
EPS = 1e-5
DEV = torch.device("cuda:0")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _nhwc(t):
    return t.to(DEV).to(torch.bfloat16).contiguous(memory_format=torch.channels_last)


def _rows(t):
    """[B,C,H,W] -> [npix, C] fp64 (pixel-major, the kernels' chunk order)."""
    return t.permute(0, 2, 3, 1).reshape(-1, t.shape[1]).double()


def _bf16_ulp(x):
    _, e = torch.frexp(x.abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(x), e - 8)


def _exact_sum_channels(Y):
    """bool [C]: fp32 accumulation of y and y^2 over the channel is exact in any order (values are multiples of q)."""
    b = Y.float().to(torch.bfloat16).view(torch.int16).int() & 0xFFFF
    man = (b & 0x7F) | 0x80
    tz = torch.log2((man & -man).float()).round().int()
    lsb = ((b >> 7) & 0xFF) - 134 + tz                                  # value is a multiple of 2^lsb
    lsb = torch.where((b & 0x7FFF) == 0, torch.full_like(lsb, 1000), lsb)
    q = torch.ldexp(torch.ones(Y.shape[1], dtype=torch.float64, device=Y.device), lsb.min(0).values.clamp(max=200))
    return (Y.abs().sum(0) < 2.0 ** 24 * q) & ((Y * Y).sum(0) < 2.0 ** 24 * q * q)


def _chain(chunks, ctas_per_sm=3):
    """Longest fp32 addition chain of a grid-stride statistics kernel over ``chunks`` 16-byte chunks."""
    grid = max(1, min(-(-chunks // 256), ctas_per_sm * _sms()))
    return -(-chunks // (256 * grid)) + 16


def bn_reference(y, gamma, beta, p, keep, cot=None, branch=None):
    """fp64 train-mode BatchNorm + LeakyReLU + Dropout of the bf16 tensor y ([B,C,H,W]) with keep mask ``keep``
    ([npix, C] bool); ``branch`` ([npix, C] bool, optional): the LeakyReLU branch to differentiate (True: positive)."""
    Y = _rows(y)
    n = Y.shape[0]
    mean = Y.mean(0)
    var = (Y - mean).square().mean(0)
    rstd = 1.0 / torch.sqrt(var + EPS)
    xhat = (Y - mean) * rstd
    g64, b64 = gamma.detach().double(), beta.detach().double()
    z = xhat * g64 + b64
    pos = z > 0 if branch is None else branch
    K = torch.ones_like(Y) if p == 0 else keep.double() * float(R.keep_scale(p))
    d = torch.where(pos, torch.ones_like(z), torch.full_like(z, SLOPE)) * K
    r = dict(Y=Y, n=n, mean=mean, var=var, rstd=rstd, xhat=xhat, z=z, pos=pos, K=K, d=d, out=z * d, gamma=g64, beta=b64)
    if cot is not None:
        G = _rows(cot)
        gp = G * d
        r.update(G=G, gp=gp, dbeta=gp.sum(0), dgamma=(gp * xhat).sum(0),
                 dy=g64 * rstd * (gp - gp.mean(0) - xhat * (gp * xhat).mean(0)))
    return r


def _bounds(r, k_stats, k_bwd, stats_rel=0.0):
    """Elementwise / per-channel error bounds for the kernel results against ``r`` (see the module docstring).
    k_stats: fp32 chain length of the batch sums ([C] or scalar; 0 = exact); k_bwd: that of the gradient sums;
    stats_rel: extra relative error of the batch sums (the conv epilogue sums its fp32 accumulator, not the bf16 y)."""
    Y, n, mean, var, rstd, g, b = r["Y"], r["n"], r["mean"], r["var"], r["rstd"], r["gamma"].abs(), r["beta"].abs()
    ka = torch.as_tensor(k_stats, dtype=torch.float64, device=Y.device) * U + stats_rel
    s1a, s2 = Y.abs().sum(0), (Y * Y).sum(0)
    dmean = ka * s1a / n + 2.0 ** -50 * mean.abs()
    dvar = 2 * ka * s2 / n + 2 * mean.abs() * dmean + 2.0 ** -48 * (var + mean * mean)
    rel_r = 0.5 * dvar / (var + EPS) + 2 * U
    dm = dmean + U * mean.abs()                                          # + rounding of mean to fp32 (save_mean)
    A = g * rstd
    ez = A * ((Y - mean).abs() * rel_r + dm) + 8 * U * (Y.abs() * A + mean.abs() * A + b)
    kink = r["z"].abs() <= ez
    out = r["out"]
    e_out = _bf16_ulp(out) + r["d"].abs() * ez + 4 * U * out.abs()
    res = dict(ez=ez, kink=kink, e_out=e_out, dmean=dm, dvar=dvar,
               rel_r=rel_r)
    if "gp" not in r:
        return res
    gp, G, K = r["gp"], r["G"], r["K"]
    flip = (1 - SLOPE) * (G * K).abs() * (kink & (r.get("branch_given") is None))   # a kink element may take either branch
    kb = k_bwd * U + 3 * U
    d_sg = kb * gp.abs().sum(0) + flip.sum(0)
    d_sgy = kb * (gp * Y).abs().sum(0) + (flip * Y.abs()).sum(0)
    sg, sgxm = r["dbeta"], (gp * (Y - mean)).sum(0)
    e_dbeta = d_sg + U * sg.abs()
    e_dg_raw = rstd * (rel_r * sgxm.abs() + d_sgy + (mean.abs() + dm) * d_sg + dm * sg.abs())
    e_dgamma = e_dg_raw + 2 * U * r["dgamma"].abs()
    mg, mgx = sg / n, r["dgamma"] / n
    dmg, dmgx = d_sg / n, e_dg_raw / n
    Yc = (Y - mean).abs()
    e_dy = (gp.abs() * A * (rel_r + 4 * U) + A * dmg + A * rstd * Yc * dmgx
            + A * mgx.abs() * (2 * rel_r * Yc + rstd * dm)
            + 4 * U * ((Y.abs() + mean.abs()) * A * rstd * (mgx.abs() + dmgx) + A * (mg.abs() + dmg) + gp.abs() * A))
    e_dy = e_dy + _bf16_ulp(r["dy"]) + 4 * U * r["dy"].abs()
    res.update(e_dbeta=e_dbeta, e_dgamma=e_dgamma, e_dy=e_dy)
    return res


def _make_bn(C, gen, rm=True):
    bn = torch.nn.BatchNorm2d(C).to(DEV)
    with torch.no_grad():
        bn.weight.copy_(1 + 0.25 * torch.randn(C, generator=gen))
        bn.bias.copy_(0.3 * torch.randn(C, generator=gen))
        if rm:
            bn.running_mean.copy_(torch.randn(C, generator=gen))
            bn.running_var.copy_(0.5 + torch.rand(C, generator=gen))
    return bn


def _run(y, bn, p, seed, cot, **kw):
    """Kernel forward + backward of bn_lrelu_dropout on y; returns out, dy, dgamma, dbeta and the running stats before."""
    from uaps_b200.bn_act import bn_lrelu_dropout
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    yk = y.detach().clone().requires_grad_(True)
    out = bn_lrelu_dropout(yk, bn, p, seed=seed, **kw)
    out.backward(cot)
    return out.detach(), yk.grad, bn.weight.grad.clone(), bn.bias.grad.clone(), rm0, rv0


def _check(r, bd, out, dy=None, dgamma=None, dbeta=None, bn=None, rm0=None, rv0=None, max_kink=1e-3, kink_ok=None):
    """Assert every kernel result against the reference ``r`` within ``bd``; returns the worst error / bound ratios."""
    C = r["Y"].shape[1]
    O = _rows(out)
    kink = bd["kink"] if kink_ok is None else kink_ok
    assert int(kink.sum()) <= 2 + max_kink * kink.numel(), f"{int(kink.sum())} elements within the rounding bound of the kink"
    sel = ~kink
    assert torch.equal(O[r["K"] == 0], torch.zeros_like(O[r["K"] == 0])), "dropped elements must be exactly 0"
    err = (O - r["out"]).abs()
    ratio = {"out": _ratio(err[sel], bd["e_out"][sel])}
    assert ratio["out"] <= 1.0, f"forward error exceeds the bound: worst ratio {ratio['out']:.3g}"
    if dy is not None:
        D = _rows(dy)
        ratio["dy"] = _ratio((D - r["dy"]).abs()[sel], bd["e_dy"][sel])
        ratio["dgamma"] = _ratio((dgamma.double() - r["dgamma"]).abs(), bd["e_dgamma"])
        ratio["dbeta"] = _ratio((dbeta.double() - r["dbeta"]).abs(), bd["e_dbeta"])
        for k in ("dy", "dgamma", "dbeta"):
            assert ratio[k] <= 1.0, f"{k} error exceeds the bound: worst ratio {ratio[k]:.3g}"
    if bn is not None:
        n, mom = r["n"], float(bn.momentum)
        unb = r["var"] * n / (n - 1) if n > 1 else r["var"]
        want_m = (1 - mom) * rm0.double() + mom * r["mean"]
        want_v = (1 - mom) * rv0.double() + mom * unb
        e_m = mom * bd["dmean"] + 4 * U * (rm0.double().abs() + want_m.abs())
        e_v = mom * bd["dvar"] * (n / (n - 1) if n > 1 else 1.0) + 4 * U * (rv0.double().abs() + want_v.abs())
        assert ((bn.running_mean.double() - want_m).abs() <= e_m).all()
        assert ((bn.running_var.double() - want_v).abs() <= e_v).all()
    return ratio


def _ratio(err, bound):
    """max of err / bound (0 / 0 counts as 0)."""
    return (err / bound.clamp_min(1e-300)).max().item()


def _keep(seed, y, p):
    npix, C = y.shape[0] * y.shape[2] * y.shape[3], y.shape[1]
    return torch.from_numpy(R.bn_keep(seed, npix, C, p)).to(DEV)


def _standalone_case(B, C, H, W, p, seed, gen):
    y = _nhwc(torch.randn(B, C, H, W, generator=gen) * 1.7 + 0.3)
    cot = _nhwc(torch.randn(B, C, H, W, generator=gen))
    bn = _make_bn(C, gen)
    out, dy, dgm, dbt, rm0, rv0 = _run(y, bn, p, seed, cot)
    r = bn_reference(y, bn.weight, bn.bias, p, _keep(seed, y, p), cot)
    chunks = B * H * W * C // 8
    k = torch.where(_exact_sum_channels(r["Y"]), 0.0, float(_chain(chunks)))
    bd = _bounds(r, k, _chain(chunks))
    return _check(r, bd, out, dy, dgm, dbt, bn, rm0, rv0)


@pytest.mark.parametrize("C", [8, 16, 32, 64, 128, 256])
@pytest.mark.parametrize("p", [0.0, 0.05, 0.1, 0.2, 0.3, 0.5])
def test_standalone_matches_fp64_reference(C, p):
    gen = torch.Generator().manual_seed(1000 * C + int(100 * p))
    for B, H, W in ((1, 1, 1), (3, 5, 7), (2, 37, 29)):                 # ragged pixel counts, one CTA to many
        _standalone_case(B, C, H, W, p, 0xC0FFEE + C, gen)


@pytest.mark.parametrize("C,p", [(16, 0.5), (64, 0.1)])
def test_standalone_past_the_unrolled_loop_threshold(C, p):
    """npix * C/8 past (U - 1) * grid * 256 chunks of every kernel (forward: U = 4, grid = 4 SMs), with a ragged tail."""
    G = C // 8
    npix = max(8 * 256 * 256 * 2 // G, 3 * 4 * _sms() * 256 // G + 1) + 3
    assert npix * G > 3 * 4 * _sms() * 256
    gen = torch.Generator().manual_seed(C)
    ratio = _standalone_case(1, C, 1, npix, p, 12345, gen)
    assert ratio["out"] <= 1.0


def _split_sums(r, nrep, gen):
    """fp64 sums of the bf16 input (exact), split unevenly over nrep replicas: [nrep][sum | sumsq][C]."""
    Y = r["Y"]
    s = torch.stack([Y.sum(0), (Y * Y).sum(0)])                          # [2, C]
    w = torch.rand(nrep, generator=gen, dtype=torch.float64).to(DEV) ** 3
    w = w / w.sum()
    parts = s.unsqueeze(0) * w.view(-1, 1, 1)
    parts[-1] = s - parts[:-1].sum(0)
    return parts.reshape(-1).contiguous()


@pytest.mark.parametrize("nrep", [1, 8, 64])
@pytest.mark.parametrize("C,p", [(16, 0.05), (32, 0.5), (128, 0.3)])
def test_replicated_sums_match_reference(nrep, C, p):
    from uaps_b200.bn_act import bn_lrelu_dropout
    gen = torch.Generator().manual_seed(nrep * 7 + C)
    y = _nhwc(torch.randn(2, C, 19, 23, generator=gen) * 1.3 - 0.4)
    cot = _nhwc(torch.randn(2, C, 19, 23, generator=gen))
    bn = _make_bn(C, gen)
    r = bn_reference(y, bn.weight, bn.bias, p, _keep(77, y, p), cot)
    sums = _split_sums(r, nrep, gen)
    out, dy, dgm, dbt, rm0, rv0 = _run(y, bn, p, 77, cot, sums=sums, nrep=nrep)
    bd = _bounds(r, nrep * 2.0 ** -29, _chain(r["n"] * C // 8))        # fp64 recombination of the replicas only
    _check(r, bd, out, dy, dgm, dbt, bn, rm0, rv0)
    # the same tensor through the statistics pass: both within their bounds of the reference, hence of each other
    bn2 = _make_bn(C, gen)
    out2 = bn_lrelu_dropout(y, bn2, p, seed=77)
    r2 = bn_reference(y, bn2.weight, bn2.bias, p, _keep(77, y, p))
    k = torch.where(_exact_sum_channels(r2["Y"]), 0.0, float(_chain(r2["n"] * C // 8)))
    _check(r2, _bounds(r2, k, 0), out2)


def test_replica_count_is_checked():
    from uaps_b200.bn_act import bn_lrelu_dropout
    y = _nhwc(torch.randn(1, 16, 4, 4))
    bn = _make_bn(16, torch.Generator().manual_seed(0))
    with pytest.raises(RuntimeError):
        bn_lrelu_dropout(y, bn, 0.1, seed=1, sums=torch.zeros(65 * 2 * 16, dtype=torch.float64, device=DEV), nrep=65)
    with pytest.raises(RuntimeError):
        bn_lrelu_dropout(y, bn, 0.1, seed=1, sums=torch.zeros(2 * 16, dtype=torch.float64, device=DEV), nrep=0)


def _conv_ref(x, w, b):
    """fp64 3x3 conv of the bf16 input with bf16-rounded weights (the packed operand) and fp32 bias."""
    return torch.nn.functional.conv2d(x.double(), w.detach().to(torch.bfloat16).double(), b.detach().double(), padding=1)


def _check_conv(x, w, b, y):
    ref = _conv_ref(x, w, b)
    mag = torch.nn.functional.conv2d(x.double().abs(), w.detach().to(torch.bfloat16).double().abs(), b.detach().double().abs(),
                                     padding=1)
    k = w.shape[1] * 9
    assert ((y.double() - ref).abs() <= _bf16_ulp(ref) + 2 * k * U * mag).all()


# The conv epilogue sums its fp32 accumulator before the bf16 rounding of y: |acc - y| <= 2^-9 |acc|, so the sums of y
# and y^2 differ from the epilogue's by at most 2^-8 of their magnitude; the epilogue's fp32 chains are <= 2^12.
CONV_STATS_REL, CONV_CHAIN = 2.0 ** -8, 4096.0


@pytest.mark.parametrize("cout,p", [(16, 0.05), (32, 0.1)])
def test_conv_epilogue_sums(cout, p):
    from uaps_b200.bn_act import bn_lrelu_dropout
    from uaps_b200.conv import conv_bf16
    gen = torch.Generator().manual_seed(cout)
    x = _nhwc(torch.randn(2, 16, 24, 40, generator=gen))
    conv = torch.nn.Conv2d(16, cout, 3, padding=1).to(DEV)
    sums = torch.zeros(8 * 2 * cout, dtype=torch.float64, device=DEV)
    with torch.no_grad():
        y = conv_bf16(x, conv.weight, conv.bias, bias_grad=False, bn_sums=sums, bn_nrep=8)
    _check_conv(x, conv.weight, conv.bias, y)
    bn = _make_bn(cout, gen)
    cot = _nhwc(torch.randn(y.shape, generator=gen))
    out, dy, dgm, dbt, rm0, rv0 = _run(y, bn, p, 99, cot, sums=sums, nrep=8)
    r = bn_reference(y, bn.weight, bn.bias, p, _keep(99, y, p), cot)
    bd = _bounds(r, CONV_CHAIN, _chain(r["n"] * cout // 8), stats_rel=CONV_STATS_REL)
    _check(r, bd, out, dy, dgm, dbt, bn, rm0, rv0, max_kink=1e-2)


def _set_key(state, key):
    key &= R.MASK64
    state.set("key_rank", key - (1 << 64) if key >= 1 << 63 else key)


@pytest.mark.parametrize("key", [0x1234_5678_9ABC_DEF1, (1 << 64) - 3])
def test_device_resident_step_key_and_direct_grads(key):
    """Inside a device-resident iteration the mask is Philox(seed + key_rank mod 2^64), forward and backward, and the
    BatchNorm gradients are added into the existing .grad."""
    from uaps_b200.bn_act import bn_lrelu_dropout
    from uaps_b200.stepctx import DeviceStepState, StepContext
    C, p = 32, 0.3
    gen = torch.Generator().manual_seed(5)
    y = _nhwc(torch.randn(2, C, 21, 17, generator=gen))
    cot = _nhwc(torch.randn(2, C, 21, 17, generator=gen))
    bn = _make_bn(C, gen)
    g0, b0 = torch.randn(C, generator=gen).to(DEV), torch.randn(C, generator=gen).to(DEV)
    bn.weight.grad, bn.bias.grad = g0.clone(), b0.clone()
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    state = DeviceStepState(DEV, lr=0.0)
    _set_key(state, key)
    yk = y.clone().requires_grad_(True)
    with StepContext(DEV, state=state) as sc:
        out = bn_lrelu_dropout(yk, bn, p)
        assert sc._seed_calls == 1
        out.backward(cot)
    seed = 0x9E3779B97F4A7C15 & (2 ** 63 - 1)                          # StepContext.next_seed, first call
    eff = (seed + key) & R.MASK64
    r = bn_reference(y, bn.weight, bn.bias, p, _keep(eff, y, p), cot)
    k = torch.where(_exact_sum_channels(r["Y"]), 0.0, float(_chain(r["n"] * C // 8)))
    bd = _bounds(r, k, _chain(r["n"] * C // 8))
    dgamma, dbeta = bn.weight.grad - g0, bn.bias.grad - b0
    bd["e_dgamma"] = bd["e_dgamma"] + 2 * U * bn.weight.grad.double().abs()
    bd["e_dbeta"] = bd["e_dbeta"] + 2 * U * bn.bias.grad.double().abs()
    _check(r, bd, out, yk.grad, dgamma, dbeta, bn, rm0, rv0)
    assert int(bn.num_batches_tracked) == 1


def test_edge_channels_constant_and_large_offset():
    """A constant channel (var = 0), channels at mean/std ~ 100 with bf16-representable spread (the E[y^2] - mean^2
    cancellation) and ordinary channels, in one tensor."""
    C, npix = 64, 2 * 30 * 26
    gen = torch.Generator().manual_seed(11)
    Y = torch.randn(npix, C, generator=gen)
    Y[:, 0] = 1.5                                                         # constant
    Y[:, 1] = -3.0
    for c in range(2, 10):                                               # offset 100, steps of 0.5 (bf16 ulp at 64..128)
        Y[:, c] = 100.0 + 0.5 * torch.randint(-3, 4, (npix,), generator=gen).float()
    for c in range(10, 14):                                              # offset -1000 (ulp 8), spread 8..24
        Y[:, c] = -1000.0 + 8.0 * torch.randint(-3, 4, (npix,), generator=gen).float()
    y = _nhwc(Y.view(2, 30, 26, C).permute(0, 3, 1, 2))
    for p in (0.0, 0.2):
        cot = _nhwc(torch.randn(2, C, 30, 26, generator=gen))
        bn = _make_bn(C, gen)
        with torch.no_grad():                                            # offset channels: z = 0.2 + {0, +-0.5, +-1, +-1.5}
            bn.weight[2:14] = 1.0
            bn.bias[2:14] = 0.2
        out, dy, dgm, dbt, rm0, rv0 = _run(y, bn, p, 4242, cot)
        r = bn_reference(y, bn.weight, bn.bias, p, _keep(4242, y, p), cot)
        k = torch.where(_exact_sum_channels(r["Y"]), 0.0, float(_chain(npix * C // 8)))
        assert bool(k[0] == 0) and bool(k[1] == 0)
        bd = _bounds(r, k, _chain(npix * C // 8))
        _check(r, bd, out, dy, dgm, dbt, bn, rm0, rv0, max_kink=1e-3)


@pytest.mark.parametrize("p", [0.0, 0.3])
def test_kink_branch_is_the_same_in_forward_and_backward(p):
    """beta = 0 and a third of each channel's pixels exactly at its (bf16-exact, exactly summed) mean: z_ref = 0 there and
    the kernel's z is its rounding of y * sc + sh.  Whatever branch the forward took (read from the sign of its output),
    the backward kernels must differentiate the same one -- in sum(g'), sum(g' y) and every element of dy."""
    C, npix = 64, 3 * 700
    gen = torch.Generator().manual_seed(21)
    m = 0.25 * torch.randint(-20, 21, (C,), generator=gen).float()      # channel means, multiples of 0.25
    m[m == 0] = 1.25
    dlt = 0.25 * torch.randint(1, 9, (C,), generator=gen).float()
    pattern = torch.tensor([-1.0, 0.0, 1.0]).repeat(npix // 3)
    Y = m + pattern[torch.randperm(npix, generator=gen)].view(-1, 1) * dlt
    y = _nhwc(Y.view(3, 20, 35, C).permute(0, 3, 1, 2))
    cot = _nhwc(torch.randn(3, C, 20, 35, generator=gen))
    bn = _make_bn(C, gen)
    with torch.no_grad():
        bn.weight.copy_(torch.linspace(0.55, 1.45, C))                   # gamma varied over the channels
        bn.bias.zero_()
    out, dy, dgm, dbt, rm0, rv0 = _run(y, bn, p, 31337, cot)
    keep = _keep(31337, y, p)
    r0 = bn_reference(y, bn.weight, bn.bias, p, keep)
    assert _exact_sum_channels(r0["Y"]).all()
    assert torch.equal(r0["mean"], m.double().to(DEV))                   # the sums, hence the mean, are exact
    at_mean = r0["Y"] == r0["mean"]
    assert (r0["z"][at_mean] == 0).all()
    branch = torch.where(at_mean, _rows(out) > 0, r0["z"] > 0)
    r = bn_reference(y, bn.weight, bn.bias, p, keep, cot, branch=branch)
    r["branch_given"] = True
    bd = _bounds(r, 0.0, _chain(npix * C // 8))
    _check(r, bd, out, dy, dgm, dbt, bn, rm0, rv0, kink_ok=torch.zeros_like(at_mean), max_kink=1.0)


# ---- the encoder block as training runs it -------------------------------------------------------------------------
def _step_bn(y, bn, p, seed, sums, cot):
    """One teacher-forced BatchNorm step on the kernel's own input y (sums: the conv epilogue's, or None); returns
    (out, dy) of the kernel after checking them, dgamma, dbeta and the running statistics against the reference."""
    out, dy, dgm, dbt, rm0, rv0 = _run(y, bn, p, seed, cot, **({} if sums is None else dict(sums=sums, nrep=8)))
    r = bn_reference(y, bn.weight, bn.bias, p, _keep(seed, y, p), cot)
    C = y.shape[1]
    if sums is None:
        k = torch.where(_exact_sum_channels(r["Y"]), 0.0, float(_chain(r["n"] * C // 8)))
        bd = _bounds(r, k, _chain(r["n"] * C // 8))
    else:
        bd = _bounds(r, CONV_CHAIN, _chain(r["n"] * C // 8), stats_rel=CONV_STATS_REL)
    _check(r, bd, out, dy, dgm, dbt, bn, rm0, rv0, max_kink=1e-2)
    return out, dy


def _step_conv(x, conv, fused, cot):
    """One teacher-forced conv step (no bias gradient: batch-statistics BatchNorm follows): output, data and weight
    gradients against fp64 on the kernel's own input and upstream gradient; returns (y, dx, sums)."""
    from uaps_b200.conv import conv_bf16
    sums = torch.zeros(8 * 2 * conv.weight.shape[0], dtype=torch.float64, device=DEV) if fused else None
    xk = x.detach().clone().requires_grad_(True)
    conv.weight.grad = None
    y = conv_bf16(xk, conv.weight, conv.bias, bias_grad=False, **({} if sums is None else dict(bn_sums=sums, bn_nrep=8)))
    _check_conv(x, conv.weight, conv.bias, y.detach())
    if cot is None:
        return y.detach(), None, sums
    y.backward(cot)
    wb = conv.weight.detach().to(torch.bfloat16).double()
    xr = x.detach().double().requires_grad_(True)
    wr = wb.clone().requires_grad_(True)
    torch.nn.functional.conv2d(xr, wr, None, padding=1).backward(cot.double())
    ga = cot.double().abs()
    mag_dx = torch.nn.grad.conv2d_input(x.shape, wb.abs(), ga, padding=1)
    mag_dw = torch.nn.grad.conv2d_weight(x.detach().double().abs(), wb.shape, ga, padding=1)
    kx, kw = conv.weight.shape[0] * 9, x.shape[0] * x.shape[2] * x.shape[3]
    assert ((xk.grad.double() - xr.grad).abs() <= _bf16_ulp(xr.grad) + 2 * kx * U * mag_dx).all()
    assert ((conv.weight.grad.double() - wr.grad).abs() <= 2 * kw * U * mag_dw + 4 * U * wr.grad.abs()).all()
    return y.detach(), xk.grad, sums


@pytest.mark.parametrize("lvl", [1, 3])
def test_encoder_block_step_by_step(lvl, monkeypatch):
    """conv (+ epilogue sums) -> BN + LeakyReLU + Dropout -> conv (+ sums) -> BN + LeakyReLU, as UNet_UAPS._block16 runs
    a training-mode encoder level; each step against its fp64 reference on the kernel's own input, forward and backward.
    Level 1 (16 -> 32 channels) takes the conv-epilogue statistics, level 3 (64 -> 128) the statistics pass."""
    import uaps_b200.bn_act as bn_act
    from uaps_b200.unet import BN_FUSE_MAX_COUT, ENC_DROPOUT, FT_CHNS, UNet_UAPS
    torch.manual_seed(lvl)
    model = UNet_UAPS(3, 4).to(DEV).train()
    blk = model.encoder.get_submodule(f"down{lvl}").maxpool_conv.get_submodule("1")
    c0, b0, c4, b4 = (blk.conv_conv.get_submodule(n) for n in ("0", "1", "4", "5"))
    cin, cout, p = FT_CHNS[lvl - 1], FT_CHNS[lvl], ENC_DROPOUT[lvl]
    fused = cout <= BN_FUSE_MAX_COUT
    assert fused == (lvl == 1)
    state0 = {k: v.clone() for k, v in blk.state_dict().items()}
    gen = torch.Generator().manual_seed(lvl)
    B, H, W = 3, 24, 40
    x = _nhwc(torch.randn(B, cin, H, W, generator=gen))
    cot = _nhwc(torch.randn(B, cout, H, W, generator=gen))
    seed = 0x5EED_0000 + lvl
    monkeypatch.setattr(bn_act, "_next_seed", lambda: seed)

    # forward, teacher-forced: every step checked on the previous step's kernel output
    y0, _, s0 = _step_conv(x, c0, fused, None)
    a0 = _step_bn(y0, b0, p, seed, s0, _nhwc(torch.zeros(y0.shape)))[0]
    y1, _, s4 = _step_conv(a0, c4, fused, None)
    # backward, teacher-forced: every step's upstream gradient is the next step's kernel gradient
    a1, dy1 = _step_bn(y1, b4, 0.0, 0, s4, cot)
    _, da0, _ = _step_conv(a0, c4, fused, dy1)
    _, dy0 = _step_bn(y0, b0, p, seed, s0, da0)
    _step_conv(x, c0, fused, dy0)

    # the product's path returns the step-by-step result (same Philox seed)
    blk.load_state_dict(state0)
    ob = model._block16(x, blk, p, None)
    if fused:                # the conv-epilogue sums are the same every run: bit for bit
        assert torch.equal(ob.detach(), a1), "UNet_UAPS._block16 left the step-by-step path"
    else:                    # the statistics pass adds in shared memory in any order: fp32 ulps of the batch sums
        assert ((_rows(ob.detach()) - _rows(a1)).abs() <= _bf16_ulp(_rows(a1))).all()
