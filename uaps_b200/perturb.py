"""Encoder-feature perturbations of the auxiliary decoders, on the fused sm_100a kernels.

Same names and call forms as the reference (utilities/UAPS_unet.py:156-185):
``FeatureNoise(uniform_range=0.3)(x)``, ``Dropout(x, p=0.5)``, ``FeatureDropout(x)``; each also
accepts the random draw it would make (``noise=``, ``keep=``, ``u=``) so a run can be replayed
against the reference bit for bit.  Without an injected draw the kernels generate it from a
Philox counter keyed by a 64-bit seed taken from ``uaps_b200.perturb.generator`` on the host, and
the backward pass regenerates the same draw from the same seed -- no mask tensor is stored.

``perturb3`` is what ``UNet_UAPS.forward`` uses: one read of a feature map, three perturbed copies.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import _lib as L

# host-side source of Philox seeds and of FeatureDropout's u (reference: np.random global, :165)
generator = np.random.default_rng(1337)
_rank_mixed = False


def manual_seed(seed: int, rank: int = 0) -> None:
    """Re-seed the host generator.  ``rank``: each data-parallel rank must draw its own dropout masks and feature noise
    (the reference's DataParallel replicas do, UAPS_model.py:13), so multi-rank callers pass their rank."""
    global generator, _rank_mixed
    generator = np.random.default_rng([int(seed), int(rank)] if rank else int(seed))
    _rank_mixed = True


def _mix_rank_once() -> None:
    """First draw in a torch.distributed process with rank > 0 and no explicit manual_seed: fold the rank into the stream."""
    global _rank_mixed
    if _rank_mixed:
        return
    _rank_mixed = True
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_rank() > 0:
            manual_seed(1337, dist.get_rank())
    except Exception:               # noqa: BLE001 -- a seed stream, never a reason to fail
        pass


def _next_seed() -> int:
    _mix_rank_once()
    return int(generator.integers(0, 2 ** 63 - 1))


def _check(x: torch.Tensor) -> torch.Tensor:
    L.require_cuda(x)
    if x.dtype != torch.float32 or x.dim() != 4:
        raise RuntimeError("feature maps must be fp32 [B, C, H, W]")
    return x if x.is_contiguous() else x.contiguous()


class _NoiseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, noise, seed, rng):
        x = _check(x)
        y = torch.empty_like(x)
        B, chw = x.shape[0], x[0].numel()
        if noise is not None:
            noise = noise.to(device=x.device, dtype=torch.float32).contiguous()
            if noise.numel() != chw:
                raise RuntimeError("noise must have shape x.shape[1:]")
        ctx.noise, ctx.seed, ctx.rng = noise, seed, rng
        with L.on_device(x.device):
            L.check(L.lib().uaps_feature_noise(x.data_ptr(), None if noise is None else noise.data_ptr(), seed, rng,
                                               y.data_ptr(), B, chw, L.stream_ptr()), "uaps_feature_noise")
        return y

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        dx = torch.empty_like(g)
        B, chw = g.shape[0], g[0].numel()
        with L.on_device(g.device):
            L.check(L.lib().uaps_feature_noise(g.data_ptr(), None if ctx.noise is None else ctx.noise.data_ptr(),
                                               ctx.seed, ctx.rng, dx.data_ptr(), B, chw, L.stream_ptr()),
                    "uaps_feature_noise(bwd)")
        return dx, None, None, None


class FeatureNoise(nn.Module):
    """x * n + x with n ~ U(-r, r) of shape x.shape[1:], one draw shared by the batch (:172-185)."""

    def __init__(self, uniform_range: float = 0.3):
        super().__init__()
        self.uniform_range = float(uniform_range)

    def forward(self, x: torch.Tensor, noise: Optional[torch.Tensor] = None, seed: Optional[int] = None):
        if noise is None and seed is None:
            seed = _next_seed()
        return _NoiseFn.apply(x, noise, 0 if seed is None else int(seed), self.uniform_range)


class _DropoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, keep, seed, p):
        x = _check(x)
        y = torch.empty_like(x)
        if keep is not None:
            keep = keep.to(device=x.device).to(torch.uint8).contiguous()
            if keep.numel() != x.numel():
                raise RuntimeError("keep mask must have x's shape")
        ctx.keep, ctx.seed, ctx.p = keep, seed, p
        with L.on_device(x.device):
            L.check(L.lib().uaps_dropout(x.data_ptr(), None if keep is None else keep.data_ptr(), seed, p,
                                         y.data_ptr(), x.numel(), L.stream_ptr()), "uaps_dropout")
        return y

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous()
        dx = torch.empty_like(g)
        with L.on_device(g.device):
            L.check(L.lib().uaps_dropout(g.data_ptr(), None if ctx.keep is None else ctx.keep.data_ptr(), ctx.seed,
                                         ctx.p, dx.data_ptr(), g.numel(), L.stream_ptr()), "uaps_dropout(bwd)")
        return dx, None, None, None


def Dropout(x: torch.Tensor, p: float = 0.5, keep: Optional[torch.Tensor] = None, seed: Optional[int] = None):
    """F.dropout(x, p) with training=True, as the reference calls it (:156-158): always active."""
    if p == 0.0:
        return x
    if keep is None and seed is None:
        seed = _next_seed()
    return _DropoutFn.apply(x, keep, 0 if seed is None else int(seed), float(p))


def _fdrop_stats(x: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    B, C, H, W = x.shape
    attention = torch.empty((B, H, W), dtype=torch.float32, device=x.device)
    smax = torch.zeros(B, dtype=torch.int32, device=x.device)
    with L.on_device(x.device):
        L.check(L.lib().uaps_fdrop_stats(x.data_ptr(), B, C, H * W, attention.data_ptr(), smax.data_ptr(),
                                         L.stream_ptr()), "uaps_fdrop_stats")
    return attention, smax


class _FeatureDropoutFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, u):
        x = _check(x)
        B, C, H, W = x.shape
        attention, smax = _fdrop_stats(x)
        y = torch.empty_like(x)
        with L.on_device(x.device):
            L.check(L.lib().uaps_fdrop_apply(x.data_ptr(), attention.data_ptr(), smax.data_ptr(), u, y.data_ptr(),
                                             B, C, H * W, L.stream_ptr()), "uaps_fdrop_apply")
        ctx.save_for_backward(attention, smax)
        ctx.u = u
        return y

    @staticmethod
    def backward(ctx, g):
        attention, smax = ctx.saved_tensors
        g = g.contiguous()
        B, C, H, W = g.shape
        dx = torch.empty_like(g)
        with L.on_device(g.device):
            L.check(L.lib().uaps_fdrop_apply(g.data_ptr(), attention.data_ptr(), smax.data_ptr(), ctx.u, dx.data_ptr(),
                                             B, C, H * W, L.stream_ptr()), "uaps_fdrop_apply(bwd)")
        return dx, None


def FeatureDropout(x: torch.Tensor, u: Optional[float] = None):
    """Zero the pixels whose channel-mean reaches u * (per-sample max of the channel-mean), one
    u ~ U(0.7, 0.9) per call shared by the batch (:161-169); no gradient through the comparison."""
    if u is None:
        u = float(generator.uniform(0.7, 0.9))
    return _FeatureDropoutFn.apply(x, float(np.float32(u)))


class _Perturb3Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, noise, keep, seed, rng, p, u):
        x = _check(x)
        B, C, H, W = x.shape
        if noise is not None:
            noise = noise.to(device=x.device, dtype=torch.float32).contiguous()
        if keep is not None:
            keep = keep.to(device=x.device).to(torch.uint8).contiguous()
        attention, smax = _fdrop_stats(x)
        ys = [torch.empty_like(x) for _ in range(3)]
        with L.on_device(x.device):
            L.check(L.lib().uaps_perturb3(x.data_ptr(), None if noise is None else noise.data_ptr(),
                                          None if keep is None else keep.data_ptr(), seed, rng, p,
                                          attention.data_ptr(), smax.data_ptr(), u,
                                          ys[0].data_ptr(), ys[1].data_ptr(), ys[2].data_ptr(),
                                          B, C, H * W, L.stream_ptr()), "uaps_perturb3")
        ctx.save_for_backward(attention, smax)
        ctx.args = (noise, keep, seed, rng, p, u)
        return tuple(ys)

    @staticmethod
    def backward(ctx, g_noise, g_drop, g_fdrop):
        attention, smax = ctx.saved_tensors
        noise, keep, seed, rng, p, u = ctx.args
        gs = [None if g is None else g.contiguous() for g in (g_noise, g_drop, g_fdrop)]
        ref = next(g for g in gs if g is not None)
        B, C, H, W = ref.shape
        dx = torch.empty_like(ref)
        with L.on_device(ref.device):
            L.check(L.lib().uaps_perturb3_bwd(*[None if g is None else g.data_ptr() for g in gs],
                                              None if noise is None else noise.data_ptr(),
                                              None if keep is None else keep.data_ptr(), seed, rng, p,
                                              attention.data_ptr(), smax.data_ptr(), u, dx.data_ptr(),
                                              B, C, H * W, L.stream_ptr()), "uaps_perturb3_bwd")
        return dx, None, None, None, None, None, None


def perturb3(x: torch.Tensor, *, noise: Optional[torch.Tensor] = None, keep: Optional[torch.Tensor] = None,
             u: Optional[float] = None, seed: Optional[int] = None, uniform_range: float = 0.3, p: float = 0.5):
    """(FeatureNoise()(x), Dropout(x, p), FeatureDropout(x)) in one pass over x (UAPS_unet.py:227-231)."""
    if seed is None:
        seed = _next_seed()
    if u is None:
        u = float(generator.uniform(0.7, 0.9))
    return _Perturb3Fn.apply(x, noise, keep, int(seed), float(uniform_range), float(p), float(np.float32(u)))


# ---- channels-last bf16 variant (bf16 / tcgen05 model path) ------------------------------------------
class _Perturb3NhwcFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, seed, rng, p, u, seed_dev, u_dev, n_out, n_alias):
        L.require_cuda(x)
        if x.dtype != torch.bfloat16 or not x.is_contiguous(memory_format=torch.channels_last):
            raise RuntimeError("perturb3_nhwc expects a channels_last bf16 [B,C,H,W] tensor")
        B, C, H, W = x.shape
        if n_out[2]:                                         # only FeatureDropout needs the channel-mean statistics
            attention = torch.empty((B, H, W), dtype=torch.float32, device=x.device)
            smax = torch.zeros(B, dtype=torch.int32, device=x.device)
        else:
            attention = smax = torch.empty(0, dtype=torch.float32, device=x.device)
        ys = [torch.empty_like(x) if n_out[i] else None for i in range(3)]      # empty_like keeps channels_last
        lib = L.lib()
        ap, sp = (attention.data_ptr(), smax.data_ptr()) if n_out[2] else (None, None)
        with L.on_device(x.device):
            if n_out[2]:
                L.check(lib.uaps_fdrop_stats_nhwc(x.data_ptr(), B, C, H * W, ap, sp, L.stream_ptr()), "uaps_fdrop_stats_nhwc")
            L.check(lib.uaps_perturb3_nhwc(x.data_ptr(), seed, rng, p, ap, sp, u,
                                           *[None if y is None else y.data_ptr() for y in ys], B, C, H * W,
                                           seed_dev, u_dev, L.stream_ptr()), "uaps_perturb3_nhwc")
        ctx.save_for_backward(attention, smax)
        ctx.args = (seed, rng, p, u, seed_dev, u_dev, n_out[2])
        # n_alias extra outputs that ARE x (views): the unperturbed consumers of the feature map take these, so x has this
        # node as its only consumer and all of its gradient contributions are summed in the one backward kernel
        return tuple(ys) + tuple(x.view_as(x) for _ in range(n_alias))

    @staticmethod
    def backward(ctx, g_noise, g_drop, g_fdrop, *g_alias):
        attention, smax = ctx.saved_tensors
        seed, rng, p, u, seed_dev, u_dev, has_stats = ctx.args
        cl = lambda g: None if g is None else g.contiguous(memory_format=torch.channels_last)
        gs = [cl(g) for g in (g_noise, g_drop, g_fdrop)]
        extra = [cl(g) for g in g_alias if g is not None]
        while len(extra) > 2:                                 # the kernel takes two; more than that never happens in UNet_UAPS
            extra = [extra[0] + extra[1]] + extra[2:]
        extra += [None] * (2 - len(extra))
        ref = next(g for g in gs + extra if g is not None)
        B, C, H, W = ref.shape
        dx = torch.empty_like(ref)
        with L.on_device(ref.device):
            L.check(L.lib().uaps_perturb3_nhwc_bwd(*[None if g is None else g.data_ptr() for g in gs], seed, rng, p,
                                                   attention.data_ptr() if has_stats else None,
                                                   smax.data_ptr() if has_stats else None, u, dx.data_ptr(), B, C, H * W,
                                                   seed_dev, u_dev, *[None if g is None else g.data_ptr() for g in extra],
                                                   L.stream_ptr()), "uaps_perturb3_nhwc_bwd")
        return (dx,) + (None,) * 8


def perturb3_nhwc(x: torch.Tensor, *, u: Optional[float] = None, seed: Optional[int] = None,
                  uniform_range: float = 0.3, p: float = 0.5, outputs=(True, True, True), aliases: int = 0,
                  seed_dev: Optional[int] = None, u_dev: Optional[int] = None):
    """Channels-last bf16 ``perturb3``: (FeatureNoise, Dropout, FeatureDropout) of one feature map in one pass.
    ``outputs``: which of the three copies to produce (None for the others) -- a 4th / 5th auxiliary decoder (the K = 5
    ablation) calls it again for ONE more copy of the perturbation family it re-uses, with a fresh draw.
    ``aliases``: that many extra outputs that are x itself -- hand them to the UNPERTURBED consumers of x (main decoder, next
    level's max-pool) and the backward kernel sums their gradients too, instead of autograd's separate accumulation passes.
    Inside a device-resident iteration (``stepctx.current().state``) the Philox key and the threshold u come from the
    device step state; otherwise they are drawn from ``uaps_b200.perturb.generator`` on the host.
    ``seed_dev`` / ``u_dev``: device addresses of a uint64 Philox key and an fp32 threshold read by the kernel at run time
    (the key is added to ``seed``, default 0; u is replaced), so a captured graph can be replayed with fresh draws."""
    from . import stepctx
    if seed_dev is not None or u_dev is not None:
        return _Perturb3NhwcFn.apply(x, int(seed or 0), float(uniform_range), float(p), float(np.float32(u or 0.8)),
                                     seed_dev, u_dev, tuple(bool(o) for o in outputs), int(aliases))
    sc = stepctx.current()
    seed_dev = u_dev = None
    if sc is not None and sc.state is not None and seed is None and u is None:
        seed, seed_dev = sc.next_seed(), sc.state.ptr("key_rank")
        if outputs[2]:
            u, u_dev = 0.8, sc.state.ptr("u", sc.next_u_slot())
        else:
            u = 0.8                                          # unused: no FeatureDropout copy requested
    if seed is None:
        seed = _next_seed()
    if u is None:
        _mix_rank_once()
        u = float(generator.uniform(0.7, 0.9))
    return _Perturb3NhwcFn.apply(x, int(seed), float(uniform_range), float(p), float(np.float32(u)), seed_dev, u_dev,
                                 tuple(bool(o) for o in outputs), int(aliases))
