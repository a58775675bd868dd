"""The convolution and resampling kernels at the launch geometry of a training iteration: bench.py's three configurations at
their per-forward batch, where every persistent CTA loops over many work units.

The toy shapes of test_conv_gpu.py give each CTA of conv_sn_kernel / conv_igemm_persistent_kernel at most one unit (a few at
most), so the code that only runs from a CTA's second unit on -- the mixed-radix tile stepping, the TMEM accumulator double
buffer, the carries and statistics reset between SN bands, the mbarrier ring after many wraps, the deterministic split-K fold
at production split counts, the max-pool's grid-stride loop -- is only reached here.  Each layer asserts, from the plan the
library prints under UAPS_CONV_DEBUG, that it really ran with more units than CTAs.

Not reached on a B200: the `s_nt != 0` branch of the persistent kernel's tile stepping (a grid that is not a multiple of the
number of output-channel blocks).  With 148 SMs every persistent grid that loops is even, so that branch stays unverified.

References: fp32 torch (TF32 off) on the same bf16-rounded operands for the convolutions, torch's CUDA max-pool for the
max-pool (bit equality, NaN included), fp64 for the upsampling.  Every output the kernels write goes into a buffer prefilled
with NaN (or, for the accumulating weight gradient, a known value), so a unit a kernel skips cannot pass on stale memory.
"""
import re

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")
BF16_TOL, F32_TOL, WGRAD_TOL = 1e-2, 2e-3, 2e-3     # of the reference scale, as test_conv_gpu.py
WGRAD_WS_MIN = 16384                                 # conv_wgrad.cu: layers with cout * cin * ks^2 >= this fold deterministically
WGRAD_BASE = 0.75                                    # what the accumulating weight gradient starts from


def _bench_configs():
    import bench
    return bench.CONFIGS


CONFIG_NAMES = ("neu", "dagm", "kosdd2")


def _pad16(c):
    return (c + 15) // 16 * 16


# ---- the layer list, from the network itself ---------------------------------------------------------------------------
def network_layers(cin, C, K, B, H, W):
    """Distinct convolutions of UNet_UAPS(cin, C, n_aux=K-1) at batch B and input H x W, in network order.  Each entry:
    name (first module of that shape), level, cin1, cin2 (concat convs: skip | upsampled), cout, ks, H, W, role
    ('bn': feeds a train-mode BatchNorm, 'up': UpBlock's conv1x1, 'logits': out_conv)."""
    from uaps_b200.unet import UNet_UAPS
    net = UNet_UAPS(cin, C, n_aux=K - 1)
    out, seen = [], set()
    for name, m in net.named_modules():
        if not isinstance(m, nn.Conv2d):
            continue
        co, ci, ks, _ = m.weight.shape
        parts = name.split(".")
        if parts[0] == "encoder":
            level, role, concat = (0 if parts[1] == "in_conv" else int(parts[1][len("down"):])), "bn", False
        else:
            assert re.fullmatch(r"main_decoder|aux_decoder\d", parts[0]), name
            if parts[1] == "out_conv":
                level, role, concat = 0, "logits", False
            else:
                i = int(parts[1][len("up"):])
                if parts[2] == "conv1x1":
                    level, role, concat = 5 - i, "up", False
                else:
                    level, role, concat = 4 - i, "bn", parts[-1] == "0"
        cin1, cin2 = (ci // 2, ci - ci // 2) if concat else (ci, 0)
        key = (cin1, cin2, co, ks, level, role)
        if key in seen:
            continue
        seen.add(key)
        out.append(dict(name=name, level=level, cin1=cin1, cin2=cin2, cout=co, ks=ks, B=B, H=H >> level, W=W >> level,
                        role=role))
    return out


def test_layer_list_covers_the_network():
    """The list holds every conv kind the network has (encoder, concat, conv1x1, logits) at all five levels, once each."""
    c = _bench_configs()["neu"]
    layers = network_layers(c["cin"], c["C"], c["K"], c["B"], c["H"], c["W"])
    assert {L["level"] for L in layers} == set(range(5))
    assert sum(L["role"] == "logits" for L in layers) == 1 and sum(L["role"] == "up" for L in layers) == 4
    assert sum(L["cin2"] > 0 for L in layers) == 4
    assert layers[0]["cin1"] == c["cin"] and layers[0]["H"] == c["H"]
    assert len({(L["cin1"], L["cin2"], L["cout"], L["ks"], L["level"]) for L in layers}) == len(layers)


# ---- kernels into NaN-filled buffers -------------------------------------------------------------------------------------
def fprop(pc, x1, x2=None, out_nchw_f32=False, split=0, slope=1.0, bn_sums=None, bn_nrep=0):
    """PackedConv.__call__ with the same arguments, but every output tensor starts as NaN."""
    from uaps_b200 import _lib as L
    B, H, W, c1s = x1.shape
    c2s = 0 if x2 is None else x2.shape[3]
    if out_nchw_f32:
        out, ocs = torch.full((B, pc.cout, H, W), float("nan"), dtype=torch.float32, device=x1.device), 0
    else:
        ocs = _pad16(pc.cout) if not split else split
        out = torch.full((B, H, W, ocs), float("nan"), dtype=torch.bfloat16, device=x1.device)
    out2 = torch.full((B, H, W, _pad16(pc.cout) - split), float("nan"), dtype=torch.bfloat16, device=x1.device) if split else None
    x2p = None if x2 is None else x2.data_ptr()
    bias = None if pc.bias is None else pc.bias.data_ptr()
    with L.on_device(x1.device):
        if bn_sums is not None:
            L.check(L.lib().uaps_conv_fprop_bn(x1.data_ptr(), c1s, x2p, c2s, pc.packed.data_ptr(), bias, out.data_ptr(), ocs,
                                               B, H, W, pc.cin1, pc.cin2, pc.cout, pc.ks, bn_sums.data_ptr(), int(bn_nrep),
                                               L.stream_ptr()), "uaps_conv_fprop_bn")
        else:
            L.check(L.lib().uaps_conv_fprop_act(x1.data_ptr(), c1s, x2p, c2s, pc.packed.data_ptr(), bias, out.data_ptr(), ocs,
                                                int(out_nchw_f32), B, H, W, pc.cin1, pc.cin2, pc.cout, pc.ks,
                                                None if out2 is None else out2.data_ptr(),
                                                0 if out2 is None else _pad16(pc.cout) - split, split, pc.fold, float(slope),
                                                L.stream_ptr()), "uaps_conv_fprop_act")
    return out if not split else (out, out2)


def check_blocks(got, ref, tol, what):
    """got, ref: [B, C, H, W].  Every (image, 16-row band, 16-channel group) block within tol of its own reference maximum."""
    B, C, H, W = ref.shape
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = (got.float() - ref).abs()
    assert not torch.isnan(err).any(), f"{what}: {int(torch.isnan(err).sum())} outputs not written (still NaN)"
    pc, ph = (-C) % 16, (-H) % 16
    e = F.pad(err, (0, 0, 0, ph, 0, pc)).reshape(B, (C + pc) // 16, 16, (H + ph) // 16, 16, W).amax(dim=(2, 4, 5))
    s = F.pad(ref.abs(), (0, 0, 0, ph, 0, pc)).reshape(B, (C + pc) // 16, 16, (H + ph) // 16, 16, W).amax(dim=(2, 4, 5))
    bad = e > tol * s
    if bad.any():
        idx = torch.nonzero(bad)[:6].tolist()
        worst = (e / s.clamp_min(1e-30)).max().item()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} (image, row band, channel group) blocks off, "
                             f"worst {worst:.3g} of the block scale (tolerance {tol}); first {idx}")


# ---- launch plans printed under UAPS_CONV_DEBUG ------------------------------------------------------------------------
_SN = re.compile(r"conv_sn(_small)?<\d+,\d+>: per_sm (\d+) .*units (\d+)")
_PERSIST = re.compile(r"conv_persistent<\d+>: .*grid (\d+) num_tiles (\d+)")
_WGRAD = re.compile(r"wgrad \d+x\d+ cout (\d+) cin (\d+) ks (\d+): ws (\d) splits (\d+) groups (\d+) tiles/cta (\d+)")


def fprop_plan(err):
    """(kernel, units, CTAs) of the one forward-kernel launch whose plan `err` holds."""
    plans = []
    for line in err.splitlines():
        m = _SN.search(line)
        if m:
            per_sm, units = int(m.group(2)), int(m.group(3))
            plans.append(("sn_small" if m.group(1) else "sn", units, min(units, _sm_count() * per_sm)))
        m = _PERSIST.search(line)
        if m:
            plans.append(("persistent", int(m.group(2)), int(m.group(1))))
    assert len(plans) == 1, err
    return plans[0]


def _sm_count():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


@pytest.fixture
def debug_plans(monkeypatch, capfd):
    """Turns on the library's per-launch plan printing and returns a function that yields what it printed since the last
    call (the C-level stderr)."""
    monkeypatch.setenv("UAPS_CONV_DEBUG", "1")
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    monkeypatch.setattr(torch.backends.cuda.matmul, "allow_tf32", False)
    capfd.readouterr()

    def take():
        torch.cuda.synchronize()
        return capfd.readouterr().err
    return take


def _rand_nhwc(g, B, H, W, c, cp, scale):
    t = torch.randn(B, H, W, cp, generator=g, device=DEV) * scale
    t[..., c:] = 0
    return t.to(torch.bfloat16)


def run_layer(L, take, g, log):
    from uaps_b200.conv import PackedConv, conv_bf16, conv_wgrad
    from uaps_b200.unet import BN_FUSE_MAX_COUT, BN_NREP
    B, H, W, c1, c2, co, ks, role = L["B"], L["H"], L["W"], L["cin1"], L["cin2"], L["cout"], L["ks"], L["role"]
    ci, cp1, cp2, cop = c1 + c2, _pad16(c1), _pad16(c2) if c2 else 0, _pad16(co)
    tag = f"{L['name']} L{L['level']} {B}x{H}x{W} {c1}+{c2}->{co} k{ks}"
    deep = L["level"] <= 1
    # distinct inputs per image, every image at its own scale
    scale = (1.0 + torch.arange(B, device=DEV, dtype=torch.float32) / 16).view(B, 1, 1, 1)
    x1 = _rand_nhwc(g, B, H, W, c1, cp1, scale)
    x2 = _rand_nhwc(g, B, H, W, c2, cp2, scale) if c2 else None
    dy = _rand_nhwc(g, B, H, W, co, cop, scale)
    w = torch.randn(co, ci, ks, ks, generator=g, device=DEV) * (2.0 / (ci * ks * ks)) ** 0.5
    b = torch.randn(co, generator=g, device=DEV) * 0.5

    # reference: fp32 conv and its autograd on the bf16-rounded operands
    xin = x1[..., :c1] if not c2 else torch.cat([x1[..., :c1], x2[..., :c2]], dim=3)
    xr = xin.permute(0, 3, 1, 2).float().contiguous().requires_grad_(True)
    wr = w.bfloat16().float().requires_grad_(True)
    yr = F.conv2d(xr, wr, b, padding=ks // 2)
    dyr = dy[..., :co].permute(0, 3, 1, 2).float().contiguous()
    yr.backward(dyr)
    yr = yr.detach()
    del xin

    def nchw(t, c):
        return t[..., :c].permute(0, 3, 1, 2)

    def plan_check(what):
        kind, units, ctas = fprop_plan(take())
        log.append(f"{tag} {what}: {kind} {units} units / {ctas} CTAs")
        if deep:
            assert units > ctas, f"{tag} {what}: {kind} ran {units} units on {ctas} CTAs -- not the many-units-per-CTA path"
        return kind

    # forward: what training runs (bf16 NHWC, BatchNorm statistics from the epilogue for the layers in front of BatchNorm;
    # fp32 NCHW logits for out_conv), then the inference epilogue with LeakyReLU
    pc = PackedConv(w, b, cin_split=c1 if c2 else None)
    take()
    if role == "logits":
        y = fprop(pc, x1, out_nchw_f32=True)
        plan_check("fprop logits")
        check_blocks(y, yr, F32_TOL, f"{tag} fp32 logits")
    else:
        sums = None
        if role == "bn":
            sums = torch.zeros(BN_NREP * 2 * cop, dtype=torch.float64, device=DEV)
            y = fprop(pc, x1, x2, bn_sums=sums, bn_nrep=BN_NREP)
        else:
            y = fprop(pc, x1, x2)
        plan_check("fprop")
        check_blocks(nchw(y, co), yr, BF16_TOL, f"{tag} fprop")
        if sums is not None:
            tot = sums.view(BN_NREP, 2, cop).sum(0)[:, :co]
            yf = y[..., :co].double().reshape(-1, co)
            n = yf.shape[0]
            mean, var = tot[0] / n, tot[1] / n - (tot[0] / n) ** 2
            mean_ref, var_ref = yf.mean(0), yf.var(0, unbiased=False)
            assert (mean - mean_ref).abs().max().item() <= 2e-3 * yf.abs().mean().item(), f"{tag} BatchNorm mean"
            assert ((var - var_ref).abs() / var_ref).max().item() <= 2e-3, f"{tag} BatchNorm variance"
            del yf
        yl = fprop(pc, x1, x2, slope=0.01)
        plan_check("fprop leaky")
        check_blocks(nchw(yl, co), F.leaky_relu(yr, 0.01), BF16_TOL, f"{tag} fprop LeakyReLU")
        del yl

    # data gradient: the same kernels with the rotated, transposed packing; a concat conv writes two tensors
    pt = PackedConv(w, None, transpose=True)
    gxr = xr.grad
    if c2:
        ga, gb = fprop(pt, dy, split=c1)
        plan_check("dgrad split")
        check_blocks(nchw(ga, c1), gxr[:, :c1], BF16_TOL, f"{tag} dgrad skip part")
        check_blocks(nchw(gb, c2), gxr[:, c1:], BF16_TOL, f"{tag} dgrad upsampled part")
        gx_parts = (ga, gb)
    else:
        gx = fprop(pt, dy)
        plan_check("dgrad")
        check_blocks(nchw(gx, ci), gxr, BF16_TOL, f"{tag} dgrad")
        gx_parts = (gx,)

    # weight gradient: workspace mode twice (bitwise equal), atomic mode once; accumulating into a known value
    xs = [x1] + ([x2] if c2 else [])
    cin_pad = cp1 + cp2
    dws, folded = [], True
    for det in (True, True, False):
        out = torch.full((co, cin_pad, ks, ks), WGRAD_BASE, dtype=torch.float32, device=DEV)
        conv_wgrad(dy, xs, co, cin_pad, ks, out=out, deterministic=det)
        launches = [m for m in map(_WGRAD.search, take().splitlines()) if m]
        assert len(launches) == len(xs), launches
        for m in launches:
            cout_l, cin_l, ks_l, ws = (int(m.group(i)) for i in (1, 2, 3, 4))
            want = det and cout_l * cin_l * ks_l * ks_l >= WGRAD_WS_MIN
            assert ws == int(want), f"{tag} wgrad ({'workspace' if det else 'atomic'} requested): ws {ws}: {m.group(0)}"
            if det:
                folded = folded and ws == 1
                log.append(f"{tag} wgrad cin {cin_l}: ws {ws} splits {m.group(5)} tiles/cta {m.group(7)}")
        dws.append(out)
    # layers below the threshold keep the fp32-atomic epilogue even when the workspace is offered: not bit-reproducible
    if folded:
        assert torch.equal(dws[0], dws[1]), f"{tag}: workspace-mode weight gradient not bitwise reproducible"
    a, c = dws[0] - WGRAD_BASE, dws[2] - WGRAD_BASE
    torch.testing.assert_close(a, c, rtol=1e-4, atol=1e-4 * c.abs().max().item(), msg=f"{tag}: workspace vs atomic")
    # input channels: the 16-padded network input maps onto the real ones, a concat's segments sit at 0 and cp1
    real = list(range(c1)) + list(range(cp1, cp1 + c2))
    gw_ref = wr.grad
    for name_, dw in (("workspace", a), ("atomic", c)):
        got = dw[:, real]
        scale_co = gw_ref.abs().amax(dim=(1, 2, 3), keepdim=True)
        bad = (got - gw_ref).abs() > WGRAD_TOL * scale_co
        assert not bad.any(), f"{tag} wgrad ({name_}): {int(bad.sum())} weights off, first {torch.nonzero(bad)[:4].tolist()}"
    pad_ch = [i for i in range(cin_pad) if i not in set(real)]
    if pad_ch:
        assert (dws[0][:, pad_ch] == WGRAD_BASE).all(), f"{tag}: weight gradient of zero padding channels"

    # the autograd op training calls: same forward and data gradient bit for bit, weight and bias gradients to the reference
    x1v = x1.permute(0, 3, 1, 2).detach().requires_grad_(True)
    x2v = x2.permute(0, 3, 1, 2).detach().requires_grad_(True) if c2 else None
    wp, bp = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    fused = role == "bn" and co <= BN_FUSE_MAX_COUT
    s = torch.zeros(BN_NREP * 2 * cop, dtype=torch.float64, device=DEV) if fused else None
    yt = conv_bf16(x1v, wp, bp, x2=x2v, nchw_f32_out=role == "logits", bias_grad=role != "bn", bn_sums=s,
                   bn_nrep=BN_NREP if fused else 0)
    if role == "logits":
        assert torch.equal(yt, y), f"{tag}: conv_bf16 logits differ from the kernel's"
        yt.backward(dyr)
    else:
        assert torch.equal(yt.permute(0, 2, 3, 1)[..., :co], y[..., :co]), f"{tag}: conv_bf16 forward differs"
        yt.backward(dy.permute(0, 3, 1, 2))
    take()
    g1 = x1v.grad.permute(0, 2, 3, 1)
    if c2:
        assert torch.equal(g1, gx_parts[0]) and torch.equal(x2v.grad.permute(0, 2, 3, 1), gx_parts[1]), f"{tag}: conv_bf16 dgrad"
    else:
        assert torch.equal(g1[..., :ci], gx_parts[0][..., :ci]), f"{tag}: conv_bf16 dgrad"
    gw = wp.grad
    assert not ((gw - gw_ref).abs() > WGRAD_TOL * gw_ref.abs().amax(dim=(1, 2, 3), keepdim=True)).any(), f"{tag}: conv_bf16 wgrad"
    if role == "bn":
        assert torch.equal(bp.grad, torch.zeros_like(bp.grad))      # in front of train-mode BatchNorm: exactly zero
    else:
        torch.testing.assert_close(bp.grad.double(), dyr.double().sum(dim=(0, 2, 3)), rtol=1e-5, atol=1e-3,
                                   msg=f"{tag}: conv_bf16 bias gradient")


@pytest.mark.parametrize("config", CONFIG_NAMES)
def test_conv_layers_at_benchmark_shapes(config, debug_plans, capfd):
    """Every distinct conv of the network, forward + data gradient + weight gradient, back to back on one stream (so the
    weight gradient's shared workspace and its barrier counters carry over from layer to layer as in an iteration)."""
    c = _bench_configs()[config]
    g = torch.Generator(device=DEV).manual_seed(1000 + CONFIG_NAMES.index(config))
    log = []
    for L in network_layers(c["cin"], c["C"], c["K"], c["B"], c["H"], c["W"]):
        run_layer(L, debug_plans, g, log)
        torch.cuda.empty_cache()
    with capfd.disabled():
        print("\n".join([f"[{config}] launch geometry on {_sm_count()} SMs:"] + log))


# ---- max-pool -------------------------------------------------------------------------------------------------------------
def _maxpool(x, gy=None):
    """uaps_maxpool2_nhwc into a NaN-filled output: x [B,H,W,C] bf16 -> [B,H/2,W/2,C], or with gy the input gradient."""
    from uaps_b200 import _lib as L
    B, H, W, C = x.shape
    shape = (B, H // 2, W // 2, C) if gy is None else (B, H, W, C)
    out = torch.full(shape, float("nan"), dtype=torch.bfloat16, device=x.device)
    with L.on_device(x.device):
        L.check(L.lib().uaps_maxpool2_nhwc(x.data_ptr(), None if gy is None else gy.data_ptr(), out.data_ptr(), B, H, W, C,
                                           L.stream_ptr()), "uaps_maxpool2_nhwc")
    return out


def _bits_equal(got, ref):
    """Bit equality of fp32 tensors, NaN matching NaN (whatever its payload)."""
    nan_g, nan_r = torch.isnan(got), torch.isnan(ref)
    return torch.equal(nan_g, nan_r) and torch.equal(got.masked_fill(nan_g, 0).view(torch.int32),
                                                     ref.masked_fill(nan_r, 0).view(torch.int32))


@pytest.mark.parametrize("config", CONFIG_NAMES)
@pytest.mark.parametrize("values", ["normal", "ties", "nan"])
def test_maxpool_matches_torch_at_level0(config, values):
    """The level-0 max-pool of each configuration (its grid-stride loop wraps many times) against torch's CUDA max_pool2d on
    the fp32 NCHW tensor of the same values, bit for bit: random values, values quantized so that most windows tie (the
    first maximum takes the gradient), and windows holding one or more NaN (torch propagates NaN and routes the gradient by
    its own rule, which the kernel must follow)."""
    from uaps_b200.unet import FT_CHNS
    c = _bench_configs()[config]
    B, H, W, C = c["B"], c["H"], c["W"], FT_CHNS[0]
    g = torch.Generator(device=DEV).manual_seed(100 * CONFIG_NAMES.index(config) + ("normal", "ties", "nan").index(values))
    x = torch.randn(B, H, W, C, generator=g, device=DEV)
    if values == "ties":
        x = torch.randint(-2, 3, (B, H, W, C), generator=g, device=DEV).float() * 0.75
    elif values == "nan":
        x[torch.rand(B, H, W, C, generator=g, device=DEV) < 0.2] = float("nan")
    x = x.to(torch.bfloat16)
    gy = torch.randn(B, H // 2, W // 2, C, generator=g, device=DEV).to(torch.bfloat16)
    chunks = B * (H // 2) * (W // 2) * C // 8
    assert chunks > _sm_count() * 8 * 256                      # more 16-byte chunks than the capped grid has threads
    xr = x.permute(0, 3, 1, 2).float().contiguous().requires_grad_(True)
    ref = F.max_pool2d(xr, 2)
    ref.backward(gy.permute(0, 3, 1, 2).float())
    y = _maxpool(x).permute(0, 3, 1, 2).float()
    gx = _maxpool(x, gy).permute(0, 3, 1, 2).float()
    assert _bits_equal(y, ref.detach()), f"forward: {int((y != ref).sum())} outputs differ"
    assert _bits_equal(gx, xr.grad), f"backward: {int((gx != xr.grad).sum())} input gradients differ"
    if values == "nan":
        assert torch.isnan(ref).any() and not torch.isnan(xr.grad).any()


def test_maxpool_nan_windows_exhaustive():
    """Every placement of NaN in a 2x2 window (16 patterns), each beside every position of the maximum, with the reference's
    NCHW and channels-last torch kernels and the bf16 path's autograd op."""
    from uaps_b200.resample import maxpool2
    pats = []
    for nan_mask in range(16):
        for top in range(4):
            v = [1.0, 2.0, 3.0, 4.0]
            v[top], v[3] = v[3], v[top]
            pats.append([float("nan") if nan_mask >> k & 1 else v[k] for k in range(4)])
    n = len(pats)
    C = 8
    x = torch.tensor(pats, device=DEV).view(n, 1, 2, 2).expand(n, C, 2, 2).to(torch.bfloat16)   # one window per image
    gy = (torch.arange(1, n * C + 1, device=DEV, dtype=torch.float32).view(n, C, 1, 1) / 8).to(torch.bfloat16)
    refs = []
    for fmt in (torch.contiguous_format, torch.channels_last):
        xr = x.float().contiguous(memory_format=fmt).requires_grad_(True)
        r = F.max_pool2d(xr, 2)
        r.backward(gy.float().contiguous(memory_format=fmt))
        refs.append((r.detach().contiguous(), xr.grad.contiguous()))
    assert _bits_equal(refs[0][0], refs[1][0]) and _bits_equal(refs[0][1], refs[1][1])
    xo = x.contiguous(memory_format=torch.channels_last).requires_grad_(True)
    y = maxpool2(xo)
    y.backward(gy.contiguous(memory_format=torch.channels_last))
    assert _bits_equal(y.float().contiguous(), refs[0][0])
    assert _bits_equal(xo.grad.float().contiguous(), refs[0][1])


# ---- bilinear x2 upsampling --------------------------------------------------------------------------------------------
def _upsample(x, backward):
    """uaps_upsample2x_nhwc into a NaN-filled output.  Forward: x [B,H,W,C] -> [B,2H,2W,C]; backward: x is the upstream
    gradient [B,2H,2W,C] -> [B,H,W,C]."""
    from uaps_b200 import _lib as L
    B, h, w, C = x.shape
    H, W = (h, w) if not backward else (h // 2, w // 2)
    shape = (B, 2 * H, 2 * W, C) if not backward else (B, H, W, C)
    out = torch.full(shape, float("nan"), dtype=torch.bfloat16, device=x.device)
    with L.on_device(x.device):
        L.check(L.lib().uaps_upsample2x_nhwc(x.data_ptr(), out.data_ptr(), B, H, W, C, int(backward), L.stream_ptr()),
                "uaps_upsample2x_nhwc")
    return out


def _bf16_ulp(v):
    """One bf16 unit in the last place at the magnitude of v (fp64)."""
    _, e = torch.frexp(v.abs().clamp_min(2.0 ** -120))
    return torch.ldexp(torch.ones_like(v), e - 8)


def interp_matrix(n):
    """[2n, n] fp64 matrix of the x2 bilinear align_corners=True taps along one axis, with the source coordinate and the two
    weights computed in fp32 as torch's fp32 kernel and src_coord in resample_nhwc.cu compute them (r = (n-1)/(2n-1) and
    s = r * o rounded to fp32, i0 = min((int)s, n-1), l1 = s - i0, l0 = 1 - l1).  Taken in fp64 from there, the only
    rounding left to the kernel is that of its fp32 arithmetic on the values."""
    r = torch.tensor(n - 1, dtype=torch.float32) / torch.tensor(2 * n - 1, dtype=torch.float32)
    o = torch.arange(2 * n)
    s = r * o.float()
    i0 = s.long().clamp(max=n - 1)
    i1 = i0 + (i0 < n - 1).long()
    l1 = s - i0.float()
    l0 = 1 - l1
    A = torch.zeros(2 * n, n, dtype=torch.float64)
    A.index_put_((o, i0), l0.double(), accumulate=True)
    A.index_put_((o, i1), l1.double(), accumulate=True)
    return A.to(DEV)


def upsample_error_ratio(B, C, H, W, g):
    """max over outputs of |kernel - fp64| / allowed, forward and backward (<= 1 passes).  Allowed: 1 bf16 ulp of the fp64
    value (the output rounding) plus 16 * 2^-24 * sum |terms| (fp32 products and sums: 4 taps forward, 16 backward)."""
    x = (torch.randn(B, H, W, C, generator=g, device=DEV) * 3).to(torch.bfloat16)
    gy = torch.randn(B, 2 * H, 2 * W, C, generator=g, device=DEV).to(torch.bfloat16)
    Ay, Ax = interp_matrix(H), interp_matrix(W)
    xd, gyd = x.double(), gy.double()
    ref = torch.einsum("oh,bhwc,pw->bopc", Ay, xd, Ax)
    ref_abs = torch.einsum("oh,bhwc,pw->bopc", Ay, xd.abs(), Ax)
    gref = torch.einsum("oh,bopc,pw->bhwc", Ay, gyd, Ax)
    gref_abs = torch.einsum("oh,bopc,pw->bhwc", Ay, gyd.abs(), Ax)
    y = _upsample(x, False).double()
    gx = _upsample(gy, True).double()
    rf = ((y - ref).abs() / (_bf16_ulp(ref) + 16 * 2.0 ** -24 * ref_abs)).amax()
    rb = ((gx - gref).abs() / (_bf16_ulp(gref) + 16 * 2.0 ** -24 * gref_abs)).amax()
    # NaN (an output the kernel did not write) compares as a failure
    return torch.stack([rf, rb]).nan_to_num(nan=float("inf"))


def test_interp_matrix_is_torch_bilinear():
    """The fp32-coordinate matrices give torch's fp64 align_corners=True upsampling up to the fp32 coordinate rounding."""
    g = torch.Generator(device=DEV).manual_seed(3)
    for H, W in ((1, 1), (1, 7), (5, 3), (15, 40), (64, 64)):
        x = torch.randn(2, 3, H, W, generator=g, device=DEV, dtype=torch.float64)
        ref = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)
        got = torch.einsum("oh,bchw,pw->bcop", interp_matrix(H), x, interp_matrix(W))
        assert (got - ref).abs().max().item() <= 1e-5 * x.abs().max().item() * max(H, W)


@pytest.mark.parametrize("config", CONFIG_NAMES)
def test_upsample_at_network_shapes(config):
    """The four upsamplings of a decoder (after up_i.conv1x1) at the configuration's batch and sizes."""
    from uaps_b200.unet import FT_CHNS
    c = _bench_configs()[config]
    g = torch.Generator(device=DEV).manual_seed(7 + CONFIG_NAMES.index(config))
    for i in range(1, 5):
        B, C, H, W = c["B"], FT_CHNS[4 - i], c["H"] >> (5 - i), c["W"] >> (5 - i)
        r = upsample_error_ratio(B, C, H, W, g)
        assert (r <= 1).all(), (config, i, (B, C, H, W), r.tolist())


@pytest.mark.parametrize("C", [8, 24, 48])
def test_upsample_every_size_to_40(C):
    """Every H, W in 1..40 (ragged CTA tiles in x and y, the 1-pixel edge cases).  C = 24 and 48 make C/8 not a power of two,
    so the 32 chunks of a CTA straddle pixel columns (the backward's per-column weight table)."""
    g = torch.Generator(device=DEV).manual_seed(C)
    ratios = torch.empty(40, 40, 2, dtype=torch.float64, device=DEV)
    for H in range(1, 41):
        for W in range(1, 41):
            ratios[H - 1, W - 1] = upsample_error_ratio(2, C, H, W, g)
    bad = torch.nonzero(ratios > 1)
    assert bad.numel() == 0, [(h + 1, w + 1, "bwd" if d else "fwd", ratios[h, w, d].item()) for h, w, d in bad[:8].tolist()]
