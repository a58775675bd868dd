"""tcgen05 implicit-GEMM convolution: Python face of uaps_conv_* (include/uaps_b200.h).

Activations are NHWC bf16 ("channels-last") with the channel count padded to a multiple of 16;
``to_nhwc_bf16`` / ``from_nhwc`` convert from and to the reference's NCHW fp32 tensors
(utilities/UAPS_unet.py works in NCHW fp32 throughout).
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import _lib as L
from . import stepctx


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


def to_nhwc_bf16(x: torch.Tensor) -> torch.Tensor:
    """[B,C,H,W] fp32 (NCHW) -> [B,H,W,pad16(C)] bf16 with zero padding channels, one kernel."""
    L.require_cuda(x)
    B, C, H, W = x.shape
    x = x.float().contiguous()
    out = torch.empty((B, H, W, pad16(C)), dtype=torch.bfloat16, device=x.device)
    with L.on_device(x.device):
        L.check(L.lib().uaps_nchw_f32_to_nhwc_bf16(x.data_ptr(), out.data_ptr(), B, C, H, W, pad16(C), L.stream_ptr()),
                "uaps_nchw_f32_to_nhwc_bf16")
    return out


def to_nhwc_bf16_with_sums(x: torch.Tensor):
    """to_nhwc_bf16 of a tensor with <= 8 channels (the logits gradient) plus the per-channel sums over all pixels of the
    bf16 values written (fp32 [C]) -- out_conv's bias gradient -- from the same kernel."""
    L.require_cuda(x)
    B, C, H, W = x.shape
    x = x.float().contiguous()
    cp = pad16(C)
    out = torch.empty((B, H, W, cp), dtype=torch.bfloat16, device=x.device)
    nrep = L.lib().uaps_nchw_f32_to_nhwc_bf16_sums_nrep()
    sc = stepctx.current()
    sums = sc.take(nrep * cp) if sc is not None else torch.zeros(nrep * cp, dtype=torch.float64, device=x.device)
    with L.on_device(x.device):
        L.check(L.lib().uaps_nchw_f32_to_nhwc_bf16_sums(x.data_ptr(), out.data_ptr(), B, C, H, W, cp, sums.data_ptr(),
                                                        L.stream_ptr()), "uaps_nchw_f32_to_nhwc_bf16_sums")
    return out, sums.view(nrep, cp)[:, :C].sum(0).float()


def channel_sums(x_nhwc: torch.Tensor, c: int) -> torch.Tensor:
    """Per-channel sum over all pixels of a channels-last bf16 tensor (fp32 [c]): the bias gradient of a conv,
    by the BatchNorm statistics kernel (fp64 accumulation)."""
    npix, cp = x_nhwc.numel() // x_nhwc.shape[-1], x_nhwc.shape[-1]
    sc = stepctx.current()
    sums = sc.take(2 * cp) if sc is not None else torch.zeros(2 * cp, dtype=torch.float64, device=x_nhwc.device)
    with L.on_device(x_nhwc.device):
        L.check(L.lib().uaps_bn_stats_nhwc(x_nhwc.data_ptr(), npix, cp, sums.data_ptr(), sums[cp:].data_ptr(), L.stream_ptr()),
                "uaps_bn_stats_nhwc")
    return sums[:c].float()


def from_nhwc(y: torch.Tensor, c: int) -> torch.Tensor:
    """[B,H,W,Cp] bf16 -> [B,c,H,W] fp32."""
    return y[..., :c].permute(0, 3, 1, 2).float().contiguous()


# Pixel folding is implemented and parity-tested, but MEASURED SLOWER on B200 (enc0.conv2, B=64: 134 us folded F=4
# vs 95 us unfolded; profiles/r01_conv_fold.txt): the folded layer needs 74 KB of resident weights (1 CTA/SM instead
# of 4) and 4x the MMA and epilogue work per byte.  It stays off unless UAPS_CONV_FOLD=1.
_FOLD_ENABLED = os.environ.get("UAPS_CONV_FOLD", "0") == "1"


def pick_fold(cins, cout: int, ks: int, W: int) -> int:
    """Pixel-folding factor for a conv whose K segments have `cins` channels: 4 for 16-channel tensors, 2 for
    32-channel ones, when the folded layer still fits the kernel's resident-weight path (N' <= 128, <= 80 KB)."""
    if not _FOLD_ENABLED:
        return 1
    cmax = max(pad16(c) for c in list(cins) + [cout])
    for f in (4, 2):
        if cmax * f > 64 or W % (8 * f) != 0:
            continue
        n_v, k_v = f * pad16(cout), sum(f * pad16(c) for c in cins)
        if n_v <= 128 and ks * ks * n_v * k_v * 2 <= 80 * 1024:
            return f
    return 1


class PackedConv:
    """Weights of one conv layer packed into the kernel's shared-memory stage image (bf16, pre-swizzled)."""

    def __init__(self, weight: torch.Tensor, bias: Optional[torch.Tensor], cin_split=None, transpose: bool = False,
                 fold: int = 1):
        L.require_cuda(weight)
        w = weight.detach().float().contiguous()
        co, ci, ks, ks2 = w.shape
        assert ks == ks2 and ks in (1, 3)
        if transpose:                       # data-gradient conv: output channels = W's input channels
            assert cin_split is None
            self.cout, self.cin1, self.cin2 = ci, co, 0
        else:
            self.cout = co
            self.cin1, self.cin2 = (ci, 0) if cin_split is None else (cin_split, ci - cin_split)
        self.ks, self.fold, self.transpose, self.shape = ks, fold, transpose, tuple(w.shape)
        nbytes = L.lib().uaps_conv_packed_bytes(self.cout, self.cin1, self.cin2, ks, fold)
        if nbytes == 0:
            raise RuntimeError("unsupported convolution shape")
        self.packed = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        self._pack(w)
        self.bias = None if bias is None else bias.detach().float().contiguous()
        if self.bias is not None and fold > 1:                # virtual bias: one padded copy per sub-pixel
            b = torch.zeros(pad16(self.cout), dtype=torch.float32, device=w.device)
            b[:self.cout] = self.bias
            self.bias = b.repeat(fold).contiguous()

    def _pack(self, w: torch.Tensor) -> None:
        with L.on_device(w.device):
            L.check(L.lib().uaps_conv_pack_weights(w.data_ptr(), self.packed.data_ptr(), self.cout, self.cin1, self.cin2,
                                                   self.ks, int(self.transpose), self.fold, L.stream_ptr()),
                    "uaps_conv_pack_weights")

    def repack(self, weight: torch.Tensor, bias: Optional[torch.Tensor]) -> "PackedConv":
        """Pack new weights of the same shape into this layer's existing buffers (weights re-packed, bias copied), so a
        CUDA graph that reads them sees the new values on its next replay.  Unfolded layers (fold = 1) only."""
        w = weight.detach().float().contiguous()
        if tuple(w.shape) != self.shape or (bias is None) != (self.bias is None) or self.fold != 1:
            raise RuntimeError("repack needs an unfolded layer and weights of the shape it was built with")
        self._pack(w)
        if bias is not None:
            self.bias.copy_(bias.detach())
        return self

    def __call__(self, x1: torch.Tensor, x2: Optional[torch.Tensor] = None, out_nchw_f32: bool = False,
                 split: int = 0, slope: float = 1.0, bn_sums: Optional[torch.Tensor] = None, bn_nrep: int = 0):
        """split > 0: return two NHWC tensors holding output channels [0, split) and [split, cout).
        slope != 1: LeakyReLU(slope) applied to conv + bias in the kernel's epilogue.
        bn_sums (fp64, bn_nrep x 2 x pad16(cout), zeroed): the kernel also accumulates the BatchNorm batch statistics of its
        output there (uaps_conv_fprop_bn)."""
        L.require_cuda(x1)
        assert x1.dtype == torch.bfloat16 and x1.is_contiguous() and x1.dim() == 4
        B, H, W, c1s = x1.shape
        c2s = 0
        if self.cin2 > 0:
            assert x2 is not None and x2.dtype == torch.bfloat16 and x2.is_contiguous() and x2.shape[:3] == x1.shape[:3]
            c2s = x2.shape[3]
        if out_nchw_f32:
            out = torch.empty((B, self.cout, H, W), dtype=torch.float32, device=x1.device)
            ocs = 0
        else:
            ocs = pad16(self.cout) if not split else split
            # folded kernels write the padding channels (zero weights -> zeros); unfolded ones mask them
            alloc = torch.zeros if (ocs != self.cout and not split and self.fold == 1) else torch.empty
            out = alloc((B, H, W, ocs), dtype=torch.bfloat16, device=x1.device)
        out2 = torch.empty((B, H, W, pad16(self.cout) - split), dtype=torch.bfloat16, device=x1.device) if split else None
        if bn_sums is not None:
            assert not out_nchw_f32 and not split and self.fold == 1 and slope == 1.0 and ocs == pad16(self.cout)
            with L.on_device(x1.device):
                L.check(L.lib().uaps_conv_fprop_bn(x1.data_ptr(), c1s, None if x2 is None else x2.data_ptr(), c2s,
                                                   self.packed.data_ptr(), None if self.bias is None else self.bias.data_ptr(),
                                                   out.data_ptr(), ocs, B, H, W, self.cin1, self.cin2, self.cout, self.ks,
                                                   bn_sums.data_ptr(), int(bn_nrep), L.stream_ptr()), "uaps_conv_fprop_bn")
            return out
        with L.on_device(x1.device):
            L.check(L.lib().uaps_conv_fprop_act(x1.data_ptr(), c1s, None if x2 is None else x2.data_ptr(), c2s,
                                                self.packed.data_ptr(), None if self.bias is None else self.bias.data_ptr(),
                                                out.data_ptr(), ocs, int(out_nchw_f32), B, H, W, self.cin1, self.cin2,
                                                self.cout, self.ks, None if out2 is None else out2.data_ptr(),
                                                0 if out2 is None else pad16(self.cout) - split, split, self.fold,
                                                float(slope), L.stream_ptr()), "uaps_conv_fprop_act")
        return out if not split else (out, out2)


_wgrad_ws = {}
_WGRAD_WS_MIN = 64 << 20
_WGRAD_DETERMINISTIC = os.environ.get("UAPS_WGRAD_ATOMIC") is None


def _wgrad_workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Scratch of the deterministic split-K weight gradient: ONE buffer per (device, stream) serves every layer (the fold
    of the partial sums ends inside the launch, and launches of a stream are ordered).  The kernel's barrier counters live
    in its first 256 bytes: zeroed at allocation, and every launch leaves them zero."""
    key = (device.index, L.stream_ptr())
    ws = _wgrad_ws.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), _WGRAD_WS_MIN), dtype=torch.uint8, device=device)
        ws[:256].zero_()                              # only the barrier counters need to start at zero
        if len(_wgrad_ws) >= 8:
            _wgrad_ws.pop(next(iter(_wgrad_ws)))
        _wgrad_ws[key] = ws
    return ws


def conv_wgrad(dy_nhwc: torch.Tensor, xs, cout: int, cin_total: int, ks: int, out: torch.Tensor = None,
               deterministic: bool = None) -> torch.Tensor:
    """dW (fp32, torch layout [cout][cin_total][ks][ks]) of a conv whose input is the channel concat of `xs`
    (NHWC bf16 tensors, each a multiple of 16 channels) and whose output gradient is dy_nhwc.  `out`: an fp32
    tensor of that shape to ACCUMULATE into (e.g. the parameter's pre-zeroed .grad) instead of a fresh one.
    deterministic (default on; UAPS_WGRAD_ATOMIC=1 turns it off): split-K partial sums go through a workspace and are
    folded in a fixed order inside the launch instead of meeting in dW through fp32 atomics."""
    B, H, W, dcs = dy_nhwc.shape
    dw = out if out is not None else torch.zeros((cout, cin_total, ks, ks), dtype=torch.float32, device=dy_nhwc.device)
    off = 0
    det = _WGRAD_DETERMINISTIC if deterministic is None else deterministic
    lib = L.lib()
    with L.on_device(dy_nhwc.device):
        for x in xs:
            c = x.shape[3]
            ws, ws_ptr, ws_n = None, None, 0
            if det:
                need = lib.uaps_conv_wgrad_workspace_bytes(B, H, W, cout, c, ks)
                if need:
                    ws = _wgrad_workspace(dy_nhwc.device, need)
                    ws_ptr, ws_n = ws.data_ptr(), ws.numel()
            L.check(lib.uaps_conv_wgrad(dy_nhwc.data_ptr(), dcs, x.data_ptr(), c, dw.data_ptr(), B, H, W, cout, c,
                                        cin_total, off, ks, ws_ptr, ws_n, L.stream_ptr()), "uaps_conv_wgrad")
            off += c
    return dw


# ---- autograd: conv layer of the bf16 path -------------------------------------------------------
def _nhwc_view(x: torch.Tensor) -> torch.Tensor:
    """Logical NCHW channels_last bf16 tensor -> its [B,H,W,C] memory view (no copy)."""
    assert x.dtype == torch.bfloat16 and x.is_contiguous(memory_format=torch.channels_last), \
        "bf16 path tensors are channels_last"
    return x.permute(0, 2, 3, 1)


def _as_cl(y_nhwc: torch.Tensor) -> torch.Tensor:
    return y_nhwc.permute(0, 3, 1, 2)        # logical NCHW, channels_last memory


_pack_cache = {}
_scope_depth = 0


class pack_scope:
    """Within this scope (one training iteration: both forwards and the backward) a parameter is packed
    once per layout instead of once per call.  The cache is dropped when the scope exits, i.e. before the
    optimizer changes the weights -- fused optimizers update parameters in place WITHOUT bumping
    ``Tensor._version``, so a version-keyed cache across steps would silently go stale."""

    def __enter__(self):
        global _scope_depth
        _scope_depth += 1
        return self

    def __exit__(self, *exc):
        global _scope_depth
        _scope_depth -= 1
        if _scope_depth == 0:
            _pack_cache.clear()
        return False


class WeightPacker:
    """All conv layers of a model re-packed with ONE launch per iteration (uaps_conv_pack_run) instead of one launch per
    (layer, layout) -- 124 launches of 4-5 us for UNet_UAPS.

    The first iteration it sees packs layer by layer as usual and records every request; ``finalize()`` turns the record into
    a device job table; from then on ``run()`` (top of every iteration, after the optimizer has changed the weights) re-packs
    everything into the same buffers and ``get()`` only hands out the cached ``PackedConv`` objects.  Valid while the
    parameters' storage stays where it is (parameters re-homed into FlatAdam's flat buffer never move)."""

    def __init__(self):
        self.entries, self.jobs, self.table, self.total_blocks = {}, [], None, 0

    @property
    def ready(self) -> bool:
        return self.table is not None

    def get(self, weight, bias, cin_split, transpose, fold) -> "PackedConv":
        key = (id(weight), transpose, cin_split, fold)
        pc = self.entries.get(key)
        if pc is None:
            pc = PackedConv(weight, bias, cin_split=cin_split, transpose=transpose, fold=fold)
            if self.ready:
                return pc                    # a layout the recorded iteration did not use: packed on the spot, not cached
            self.entries[key] = pc
            co, ci = weight.shape[0], weight.shape[1]
            cout, cin1, cin2 = (ci, co, 0) if transpose else (co, ci if cin_split is None else cin_split,
                                                              0 if cin_split is None else ci - cin_split)
            self.jobs.append((weight.detach(), pc.packed, cout, cin1, cin2, pc.ks, int(transpose), fold))
        return pc

    def finalize(self, device: torch.device) -> None:
        if self.ready or not self.jobs:
            return
        n = len(self.jobs)
        arr = (L.PackJobStruct * n)()
        for i, (w, dst, cout, cin1, cin2, ks, tr, fold) in enumerate(self.jobs):
            if w.dtype != torch.float32 or not w.is_contiguous():
                return                       # packing goes through a converted copy: keep the per-layer path
            arr[i] = L.PackJobStruct(w.data_ptr(), dst.data_ptr(), cout, cin1, cin2, ks, tr, fold)
        import ctypes as C
        lib = L.lib()
        host = torch.empty(n * lib.uaps_conv_pack_job_bytes(), dtype=torch.uint8)
        total = C.c_int(0)
        L.check(lib.uaps_conv_pack_plan(arr, n, host.data_ptr(), C.byref(total)), "uaps_conv_pack_plan")
        self.table, self.total_blocks = host.to(device), int(total.value)

    def run(self) -> None:
        with L.on_device(self.table.device):
            L.check(L.lib().uaps_conv_pack_run(self.table.data_ptr(), len(self.jobs), self.total_blocks, L.stream_ptr()),
                    "uaps_conv_pack_run")


def packed(weight: torch.Tensor, bias, cin_split=None, transpose: bool = False, fold: int = 1) -> "PackedConv":
    sc = stepctx.current()
    if sc is not None and sc.packer is not None:
        return sc.packer.get(weight, bias, cin_split, transpose, fold)
    if _scope_depth == 0:
        return PackedConv(weight, bias, cin_split=cin_split, transpose=transpose, fold=fold)
    key = (id(weight), transpose, cin_split, fold)
    hit = _pack_cache.get(key)
    if hit is None:
        hit = PackedConv(weight, bias, cin_split=cin_split, transpose=transpose, fold=fold)
        _pack_cache[key] = hit
    return hit


class _ConvFn(torch.autograd.Function):
    """y = conv(cat([x1, x2]), W) + b on tcgen05; dX by the same kernel with the rotated/transposed
    packing; dW by the tcgen05 weight-gradient kernel (conv_wgrad.cu)."""

    @staticmethod
    def forward(ctx, x1, x2, weight, bias, nchw_f32_out, bias_grad, bn_sums, bn_nrep):
        co, ci, ks, _ = weight.shape
        c1 = x1.shape[1]
        split = None if x2 is None else c1
        W_img = x1.shape[3]
        cins = [c1] if x2 is None else [c1, x2.shape[1]]
        conv = packed(weight, bias, cin_split=split, fold=pick_fold(cins, co, ks, W_img))
        y = conv(_nhwc_view(x1), None if x2 is None else _nhwc_view(x2), out_nchw_f32=nchw_f32_out, bn_sums=bn_sums, bn_nrep=bn_nrep)
        ctx.save_for_backward(x1, x2, weight)
        ctx.has_bias, ctx.nchw, ctx.bias_grad = bias is not None, nchw_f32_out, bias_grad
        ctx.weight_param = weight
        return y if nchw_f32_out else _as_cl(y)

    @staticmethod
    def backward(ctx, gy):
        x1, x2, weight = ctx.saved_tensors
        co, ci, ks, _ = weight.shape
        gb_fused = None
        if ctx.nchw:                                         # fp32 NCHW logits gradient -> bf16 channels-last, 16-padded
            if ctx.has_bias and ctx.bias_grad and co <= 8:   # ... and out_conv's bias gradient from the same pass
                gy_nhwc, gb_fused = to_nhwc_bf16_with_sums(gy)
            else:
                gy_nhwc = to_nhwc_bf16(gy)
        else:
            if not gy.is_contiguous(memory_format=torch.channels_last):
                gy = gy.contiguous(memory_format=torch.channels_last)
            gy_nhwc = gy.permute(0, 2, 3, 1)
            if gy_nhwc.shape[-1] % 16:                        # pad the K segment to the kernel's granule
                pad = torch.zeros((*gy_nhwc.shape[:3], pad16(co)), dtype=torch.bfloat16, device=gy.device)
                pad[..., :co] = gy_nhwc
                gy_nhwc = pad
        # data gradient: tcgen05 kernel, W'[ci][co] rotated by 180 degrees
        c1 = x1.shape[1]
        fold = pick_fold([co], ci if x2 is None else pad16(ci), ks, gy_nhwc.shape[2])
        if x2 is None:
            gx = packed(weight, None, transpose=True, fold=fold)(gy_nhwc)   # [B,H,W,pad16(ci)]
            g1 = _as_cl(gx[..., :c1]) if ctx.needs_input_grad[0] else None
            g2 = None
        else:                                                            # concat conv: each consumer gets its own tensor
            ga, gb2 = packed(weight, None, transpose=True, fold=fold)(gy_nhwc, split=c1)
            g1 = _as_cl(ga) if ctx.needs_input_grad[0] else None
            g2 = _as_cl(gb2) if ctx.needs_input_grad[1] else None
        # weight gradient: tcgen05 kernel on the same channels-last tensors (MN-major operands, no transposes)
        xs = [_nhwc_view(x1)] + ([] if x2 is None else [_nhwc_view(x2)])
        cin_pad = sum(t.shape[3] for t in xs)                 # the 3-channel network input is stored 16-padded
        sc = stepctx.current()
        wparam = ctx.weight_param
        direct = (sc is not None and sc.direct_grads and cin_pad == ci and wparam.grad is not None
                  and wparam.grad.dtype == torch.float32 and wparam.grad.is_contiguous())
        if direct:                               # accumulate straight into the pre-zeroed .grad view
            conv_wgrad(gy_nhwc, xs, co, cin_pad, ks, out=wparam.grad)
            gw = None
        else:
            gw = conv_wgrad(gy_nhwc, xs, co, cin_pad, ks)
            if cin_pad != ci:
                gw = gw[:, :ci].contiguous()
        gb = None
        if ctx.has_bias:
            # a bias in front of train-mode BatchNorm has an analytically zero gradient; only conv1x1 /
            # out_conv (bias_grad=True) need the reduction
            if ctx.bias_grad:
                gb = gb_fused if gb_fused is not None else channel_sums(gy_nhwc, co)
            elif not direct:
                gb = torch.zeros(co, dtype=torch.float32, device=gy.device)
        return g1, g2, gw, gb, None, None, None, None


def conv_bf16(x1: torch.Tensor, weight: torch.Tensor, bias, x2: torch.Tensor = None, nchw_f32_out: bool = False,
              bias_grad: bool = True, bn_sums: torch.Tensor = None, bn_nrep: int = 0):
    """bias_grad=False: the conv feeds a train-mode BatchNorm, whose mean subtraction makes d loss / d bias
    exactly zero -- the reduction is skipped and zeros are returned (the reference accumulates rounding noise).
    bn_sums / bn_nrep: also accumulate the batch statistics of the output for that BatchNorm (see PackedConv.__call__)."""
    return _ConvFn.apply(x1, x2, weight, bias, nchw_f32_out, bias_grad, bn_sums, bn_nrep)
