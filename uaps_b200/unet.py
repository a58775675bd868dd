"""Drop-in UAPS multi-decoder U-Net (utilities/UAPS_unet.py:208-233) on the B200 kernels.

``UNet_UAPS(in_chns, class_num)`` keeps the reference's constructor, its 4-tuple output
``(main, aux1, aux2, aux3)`` of [B, C, H, W] fp32 logits, and -- key for key, 334 tensors -- its
``state_dict`` (e.g. ``encoder.down2.maxpool_conv.1.conv_conv.4.weight``,
``aux_decoder3.up1.conv1x1.bias``), so reference checkpoints load unchanged (with or without the
``module.`` prefix DataParallel adds, see ``load_reference_state_dict``).

Internally it is not a module-per-layer tree: parameters sit in holder modules that only give
them their reference names, and ``forward`` is a straight-line program.  The three auxiliary
perturbations of all five encoder levels (reference :227-231: 15 tensors, ~40 ATen launches, a CPU
RNG draw plus an H2D copy per level) are one fused kernel per level (``perturb.perturb3``), the
encoder-block dropout (:40) is the Philox dropout kernel.

Layer semantics kept from the reference (SURVEY.md Q1-Q3, Q14): the up path is conv1x1 +
bilinear(align_corners=True) because ``UpBlock``'s ``bilinear=True`` default wins (:69);
``F.dropout`` of aux2 is active in eval mode too (:156-158); H and W must be multiples of 16.
"""
from __future__ import annotations

import re
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from . import perturb as P
from .bn_act import bn_lrelu_dropout
from .conv import PackedConv, conv_bf16, pad16, to_nhwc_bf16
from .resample import maxpool2, upsample2x

FT_CHNS = (16, 32, 64, 128, 256)            # UAPS_unet.py:212
ENC_DROPOUT = (0.05, 0.1, 0.2, 0.3, 0.5)    # :214
_AUX_KINDS = ("noise", "dropout", "fdrop")  # :227, :229, :231; a 4th/5th aux decoder re-uses them in order
BN_NREP = 8                                 # replicas of the BatchNorm sums a conv epilogue accumulates into (spreads the atomics)
BN_FUSE_MAX_COUT = int(__import__("os").environ.get("UAPS_BN_FUSE_MAX_COUT", "32"))   # widest layer whose conv epilogue takes the statistics


def _check_hw(x: torch.Tensor) -> None:
    if x.shape[-1] % 16 or x.shape[-2] % 16:
        raise RuntimeError("H and W must be multiples of 16 (four 2x poolings; the reference fails in torch.cat)")


def _holder(**children: nn.Module) -> nn.Module:
    m = nn.Module()
    for name, child in children.items():
        m.add_module(name, child)
    return m


def _conv_block(cin: int, cout: int) -> nn.Module:
    """Parameters of ConvBlock (:31-47) under its Sequential indices 0 (conv), 1 (BN), 4 (conv), 5 (BN)."""
    return _holder(conv_conv=_holder(**{
        "0": nn.Conv2d(cin, cout, kernel_size=3, padding=1), "1": nn.BatchNorm2d(cout),
        "4": nn.Conv2d(cout, cout, kernel_size=3, padding=1), "5": nn.BatchNorm2d(cout)}))


def _encoder(in_chns: int) -> nn.Module:
    enc = _holder(in_conv=_conv_block(in_chns, FT_CHNS[0]))
    for lvl in range(1, 5):                                   # DownBlock (:50-62): MaxPool2d is child "0", block is "1"
        enc.add_module(f"down{lvl}", _holder(maxpool_conv=_holder(**{"1": _conv_block(FT_CHNS[lvl - 1], FT_CHNS[lvl])})))
    return enc


def _decoder(class_num: int) -> nn.Module:
    dec = nn.Module()
    for i in range(1, 5):                                     # UpBlock (:65-86), channels :129-136
        c1, c2 = FT_CHNS[5 - i], FT_CHNS[4 - i]
        dec.add_module(f"up{i}", _holder(conv1x1=nn.Conv2d(c1, c2, kernel_size=1), conv=_conv_block(2 * c2, c2)))
    dec.add_module("out_conv", nn.Conv2d(FT_CHNS[0], class_num, kernel_size=3, padding=1))
    return dec


class UNet_UAPS(nn.Module):
    def __init__(self, in_chns: int, class_num: int, n_aux: int = 3, compute: str = "bf16"):
        super().__init__()
        if not 0 <= n_aux <= 5:
            raise ValueError("n_aux must be in [0, 5]")
        if compute == "reference":
            compute = "fp32"
        if compute not in ("fp32", "bf16"):
            raise ValueError("compute must be 'bf16' (default), or 'fp32' / 'reference'")
        self.in_chns, self.class_num, self.n_aux = in_chns, class_num, n_aux
        # "bf16" (default, the product path): channels-last bf16 activations, every layer a hand-written sm_100a
        #         kernel (tcgen05 implicit-GEMM fprop / dgrad / wgrad, fused BN, resampling, Philox perturbations),
        #         fp32 master weights and accumulation, 1e-2 parity.
        # "fp32" / "reference": every layer in fp32 NCHW through torch (cuDNN) -- kept ONLY as the
        #         reference-precision path for parity runs against the reference's golden vectors (1e-4).
        self.compute = compute
        self.encoder = _encoder(in_chns)
        self.main_decoder = _decoder(class_num)
        for a in range(1, n_aux + 1):
            self.add_module(f"aux_decoder{a}", _decoder(class_num))

    # ---- layers -----------------------------------------------------------------------------
    def _block(self, x: torch.Tensor, blk: nn.Module, p_drop: float, keep, seed) -> torch.Tensor:
        cc = blk.conv_conv
        y = F.leaky_relu(cc.get_submodule("1")(cc.get_submodule("0")(x)), 0.01)
        if p_drop > 0.0 and self.training:                    # nn.Dropout(p) between the two convs (:40)
            y = P.Dropout(y, p_drop, keep=keep, seed=seed)
        return F.leaky_relu(cc.get_submodule("5")(cc.get_submodule("4")(y)), 0.01)

    def encode(self, x: torch.Tensor, enc_keep: Optional[Sequence[torch.Tensor]] = None) -> List[torch.Tensor]:
        """Encoder.forward (:110-116): five levels, MaxPool2d(2) in front of levels 1-4."""
        feats = []
        for lvl in range(5):
            if lvl == 0:
                blk = self.encoder.in_conv
            else:
                x = F.max_pool2d(x, 2)
                blk = self.encoder.get_submodule(f"down{lvl}").maxpool_conv.get_submodule("1")
            x = self._block(x, blk, ENC_DROPOUT[lvl], None if enc_keep is None else enc_keep[lvl], None)
            feats.append(x)
        return feats

    def decode(self, feats: Sequence[torch.Tensor], dec: nn.Module) -> torch.Tensor:
        """Decoder.forward (:141-153) with UpBlock.forward (:81-86)."""
        x = feats[4]
        for i in range(1, 5):
            up = dec.get_submodule(f"up{i}")
            x = up.conv1x1(x)
            x = F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True)
            x = torch.cat([feats[4 - i], x], dim=1)
            x = self._block(x, up.conv, 0.0, None, None)
        return dec.out_conv(x)

    # ---- bf16 / tcgen05 path ------------------------------------------------------------------
    @staticmethod
    def _bn_sums(cout: int, device) -> torch.Tensor:
        """Zeroed fp64 [BN_NREP][sum | sumsq][pad16(cout)] for the conv epilogue's BatchNorm statistics."""
        from . import stepctx
        n = BN_NREP * 2 * pad16(cout)
        sc = stepctx.current()
        return sc.take(n) if sc is not None else torch.zeros(n, dtype=torch.float64, device=device)

    def _block16(self, x, blk, p_drop, keep, x2=None):
        cc = blk.conv_conv
        c0, b0, c4, b4 = (cc.get_submodule(n) for n in ("0", "1", "4", "5"))
        # a conv bias in front of a BatchNorm that uses BATCH statistics has an analytically zero gradient; with running
        # statistics (eval mode, e.g. fine-tuning with frozen BN) it does not
        bg = not self.training
        if self.training and keep is None:
            # conv (its epilogue also accumulates the BatchNorm batch statistics) -> fused BN(batch stats) + LeakyReLU +
            # Philox dropout: 2 kernels per layer forward, 2 + dgrad + wgrad backward
            # The epilogue statistics cost the conv ~150 instructions per 32 x 16 accumulator fragment.  Measured (B = 64): for the
            # 16/32-channel layers that is +5..18 us on the conv against 16..29 us for the separate statistics pass it replaces;
            # for 64+ channels (8 fragments per tile, small tensors) it costs more than the 8 us pass -> those keep bn_stats.
            cout = c0.weight.shape[0]
            if cout <= BN_FUSE_MAX_COUT:
                s0, s4 = self._bn_sums(cout, x.device), self._bn_sums(cout, x.device)
                y = conv_bf16(x, c0.weight, c0.bias, x2=x2, bias_grad=bg, bn_sums=s0, bn_nrep=BN_NREP)
                y = bn_lrelu_dropout(y, b0, p_drop, sums=s0, nrep=BN_NREP)
                y = conv_bf16(y, c4.weight, c4.bias, bias_grad=bg, bn_sums=s4, bn_nrep=BN_NREP)
                return bn_lrelu_dropout(y, b4, 0.0, sums=s4, nrep=BN_NREP)
            y = bn_lrelu_dropout(conv_bf16(x, c0.weight, c0.bias, x2=x2, bias_grad=bg), b0, p_drop)
            return bn_lrelu_dropout(conv_bf16(y, c4.weight, c4.bias, bias_grad=bg), b4, 0.0)
        y = conv_bf16(x, c0.weight, c0.bias, x2=x2, bias_grad=bg)
        y = F.leaky_relu(b0(y), 0.01)                         # eval mode / injected dropout mask (parity runs)
        if p_drop > 0.0 and self.training:
            y = y * (keep.to(y.dtype) * (1.0 / (1.0 - p_drop)))
        return F.leaky_relu(b4(conv_bf16(y, c4.weight, c4.bias, bias_grad=bg)), 0.01)

    def _encode16(self, x, enc_keep, perturbed=None):
        """perturbed: a list to receive, per level, the (noise, dropout, feature-dropout) copies of the level's feature map
        (rows a2-a4, one fused Philox kernel per level).  The unperturbed consumers of the feature map -- the main decoder
        and the next level's max-pool -- then take ALIAS outputs of that kernel's autograd node, so the feature map's whole
        gradient (three perturbed decoders + main decoder + pool) is summed by the one backward kernel instead of by
        autograd's separate accumulation passes."""
        B, C, H, W = x.shape
        x16 = to_nhwc_bf16(x).permute(0, 3, 1, 2)             # logical NCHW, channels-last memory, 16-padded
        feats, cur = [], x16
        live = tuple(a <= self.n_aux for a in (1, 2, 3))
        for lvl in range(5):
            if lvl == 0:
                blk = self.encoder.in_conv
            else:
                cur = maxpool2(cur)
                blk = self.encoder.get_submodule(f"down{lvl}").maxpool_conv.get_submodule("1")
            cur = self._block16(cur, blk, ENC_DROPOUT[lvl], None if enc_keep is None else enc_keep[lvl])
            if perturbed is not None:
                outs = P.perturb3_nhwc(cur, outputs=live, aliases=2 if lvl < 4 else 1)
                perturbed.append(outs[:3])
                feats.append(outs[3])                          # for the main decoder
                cur = outs[4] if lvl < 4 else outs[3]          # for the next level's max-pool
            else:
                feats.append(cur)
        return feats

    def _decode16(self, feats, dec):
        x = feats[4]
        for i in range(1, 5):
            up = dec.get_submodule(f"up{i}")
            x = upsample2x(conv_bf16(x, up.conv1x1.weight, up.conv1x1.bias))
            x = self._block16(feats[4 - i], up.conv, 0.0, None, x2=x)           # concat as two K segments
        return conv_bf16(x, dec.out_conv.weight, dec.out_conv.bias, nchw_f32_out=True)

    def _forward16(self, x, rand):
        fused = [] if (rand is None and self.n_aux > 0) else None     # one fused Philox kernel per level (rows a2-a4)
        feats = self._encode16(x, None if rand is None else rand["enc_keep"], perturbed=fused)
        outs = [self._decode16(feats, self.main_decoder)]
        for a in range(1, self.n_aux + 1):
            kind = _AUX_KINDS[(a - 1) % 3]
            if fused is not None and a <= 3:
                outs.append(self._decode16([t[a - 1] for t in fused], self.get_submodule(f"aux_decoder{a}")))
                continue
            if rand is None:
                # 4th / 5th auxiliary decoder (the K = 5 ablation; the reference has only commented ``aux4`` stubs,
                # UAPS_train.py:139,182,190, so the perturbation is this repo's choice: the same three families in
                # order, with a fresh draw): the same kernel, asked for the one copy it needs
                sel = tuple(k == kind for k in _AUX_KINDS)
                pf = [P.perturb3_nhwc(f, outputs=sel)[_AUX_KINDS.index(kind)] for f in feats]
                outs.append(self._decode16(pf, self.get_submodule(f"aux_decoder{a}")))
                continue
            pf = []
            for lvl, f in enumerate(feats):                    # injected draws (parity runs only): torch expressions
                if kind == "noise":
                    n = rand["noise"][lvl].to(f.dtype)
                    pf.append(f * n.unsqueeze(0) + f)
                elif kind == "dropout":
                    pf.append(f * (rand["aux2_keep"][lvl].to(f.dtype) * 2.0))
                else:
                    u = rand["u"][lvl]
                    att = f.float().mean(dim=1, keepdim=True)
                    thr = att.flatten(1).max(dim=1)[0].view(-1, 1, 1, 1) * u
                    pf.append(f * (att < thr).to(f.dtype))
            outs.append(self._decode16(pf, self.get_submodule(f"aux_decoder{a}")))
        return tuple(outs) if self.n_aux else outs[0]

    # ---- inference: BatchNorm folded into the convolutions, LeakyReLU in the conv epilogue --------------------
    @staticmethod
    def _fold_bn(conv: nn.Conv2d, bn: nn.BatchNorm2d):
        """Eval-mode BN(conv(x)) as one convolution: w' = w * g / sqrt(var + eps), b' = (b - mean) * g / sqrt(var + eps) + beta."""
        s = bn.weight.detach().float() * torch.rsqrt(bn.running_var.detach().float() + bn.eps)
        w = conv.weight.detach().float() * s.view(-1, 1, 1, 1)
        b = (conv.bias.detach().float() - bn.running_mean.detach().float()) * s + bn.bias.detach().float()
        return w.contiguous(), b.contiguous()

    def _block_plan(self, blk, cin_split=None, make=PackedConv):
        cc = blk.conv_conv
        w0, b0 = self._fold_bn(cc.get_submodule("0"), cc.get_submodule("1"))
        w4, b4 = self._fold_bn(cc.get_submodule("4"), cc.get_submodule("5"))
        return make(w0, b0, cin_split=cin_split), make(w4, b4)

    def _decoder_plan(self, dm: nn.Module, make=PackedConv):
        dec = []
        for i in range(1, 5):
            up = dm.get_submodule(f"up{i}")
            c2 = FT_CHNS[4 - i]
            dec.append((make(up.conv1x1.weight, up.conv1x1.bias), *self._block_plan(up.conv, cin_split=c2, make=make)))
        return dec, make(dm.out_conv.weight, dm.out_conv.bias)

    def _main_plan(self, make=PackedConv):
        """(enc, dec, out): the BN-folded layers of encoder + main decoder, each built by ``make(weight, bias,
        cin_split=None)`` in a fixed order (``validate.Validator`` re-packs its own copy in place through it)."""
        enc = [self._block_plan(self.encoder.in_conv, make=make)] + \
              [self._block_plan(self.encoder.get_submodule(f"down{lvl}").maxpool_conv.get_submodule("1"), make=make)
               for lvl in range(1, 5)]
        dec, out = self._decoder_plan(self.main_decoder, make=make)
        return enc, dec, out

    def _inference_plan(self):
        """Packed, BN-folded layers of encoder + main decoder (built lazily, dropped by train() / load_state_dict()), and
        a dict that receives the auxiliary decoders' layers when an ensemble first needs them (``_aux_plan``)."""
        plan = getattr(self, "_infer_plan", None)
        if plan is not None:
            return plan
        self._infer_plan = (*self._main_plan(), {})
        return self._infer_plan

    def _aux_plan(self, a: int):
        aux = self._inference_plan()[3]
        if a not in aux:
            aux[a] = self._decoder_plan(self.get_submodule(f"aux_decoder{a}"))
        return aux[a]

    @staticmethod
    def _encode_folded(x, enc):
        """Folded encoder: five levels of channels-last bf16 feature maps [B,H_l,W_l,C_l]."""
        cur = to_nhwc_bf16(x)                                                # [B,H,W,16]
        feats = []
        for lvl, (c0, c4) in enumerate(enc):
            if lvl:
                cur = maxpool2(cur.permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
            cur = c4(c0(cur, slope=0.01), slope=0.01)
            feats.append(cur)
        return feats

    @staticmethod
    def _decode_folded(feats, dec, out):
        """Folded decoder over channels-last feature maps: fp32 NCHW logits."""
        cur = feats[4]
        for i, (c1x1, c0, c4) in enumerate(dec, start=1):
            up = upsample2x(c1x1(cur).permute(0, 3, 1, 2)).permute(0, 2, 3, 1)
            cur = c4(c0(feats[4 - i], up, slope=0.01), slope=0.01)
        return out(cur, out_nchw_f32=True)

    def train(self, mode: bool = True):
        self._infer_plan = None                       # weights are about to change: drop the folded copies
        self.__dict__.pop("_graphs", None)
        return super().train(mode)

    def load_state_dict(self, *args, **kw):
        self._infer_plan = None
        self.__dict__.pop("_graphs", None)
        return super().load_state_dict(*args, **kw)

    @torch.no_grad()
    def predict(self, x: torch.Tensor) -> torch.Tensor:
        """Validation / inference fast path (UAPS_train.py:377, UAPS-Testing.ipynb): the main decoder's logits only.
        The reference runs -- and perturbs -- all three auxiliary decoders here and throws their outputs away.

        bf16 path in eval mode: BatchNorm's running statistics are folded into the conv weights and LeakyReLU runs in
        the conv epilogue (``uaps_conv_fprop_act``), so the whole forward is 23 tcgen05 conv launches, 4 max-pools and
        4 upsamples -- no BatchNorm or activation pass touches HBM.  In training mode (batch statistics) and on the
        fp32 path it falls back to the ordinary layers."""
        if self.compute == "bf16" and not self.training:
            enc, dec, out, _ = self._inference_plan()
            return self._decode_folded(self._encode_folded(x, enc), dec, out)
        if self.compute == "bf16":
            return self._decode16(self._encode16(x, None), self.main_decoder)
        return self.decode(self.encode(x), self.main_decoder)

    @torch.no_grad()
    def predict_graphed(self, x: torch.Tensor) -> torch.Tensor:
        """``predict`` replayed from a CUDA graph (bf16 path, eval mode): the ~31 launches of a forward are captured once
        per input shape and replayed with one ``cudaGraphLaunch``, which is what latency-bound serving (batch 1: the
        forward is ~35 launches of a few microseconds each) needs.  The returned tensor is the graph's static output
        buffer: it is overwritten by the next call with the same shape (clone it to keep it)."""
        if self.compute != "bf16" or self.training:
            return self.predict(x)
        key = (tuple(x.shape), x.device.index)
        cache = self.__dict__.setdefault("_graphs", {})
        entry = cache.get(key)
        if entry is None or entry[3] is not self._inference_plan():
            static_in = torch.empty_like(x, dtype=torch.float32)
            static_in.copy_(x)
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(torch.cuda.current_stream(x.device))
            with torch.cuda.stream(side):                       # warm-up off the capture: lazy inits, plan, allocator
                for _ in range(2):
                    self.predict(static_in)
            torch.cuda.current_stream(x.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = self.predict(static_in)
            entry = (graph, static_in, static_out, self._inference_plan())
            cache[key] = entry
        graph, static_in, static_out, _ = entry
        static_in.copy_(x)
        graph.replay()
        return static_out

    # ---- ensemble inference: every decoder, label map + uncertainty maps (DESIGN.md f5) -------------------------------
    def _ensemble_calls(self) -> int:
        """Perturbation launches of an ensemble forward: one per level for auxiliary decoders 1-3 together, then one per
        level for each of decoders 4 and 5."""
        return 5 * (1 + max(0, self.n_aux - 3))

    def _ensemble_draws(self, seed: Optional[int]) -> np.ndarray:
        """Host int64 [2, n]: row 0 the Philox keys, row 1 the FeatureDropout thresholds (fp32 in the low 4 bytes), one
        column per perturbation launch (see ``predict_uncertainty`` for the order)."""
        if seed is None:
            P._mix_rank_once()
            rng = P.generator
        else:
            rng = np.random.default_rng(int(seed))
        n = self._ensemble_calls()
        draws = np.zeros((2, n), dtype=np.int64)
        u32 = draws[1].view(np.float32)                       # little-endian: float i sits at index 2i
        for i in range(n):
            draws[0, i] = rng.integers(0, 2 ** 63 - 1)
            u32[2 * i] = rng.uniform(0.7, 0.9)
        return draws

    def _ensemble_logits16(self, x: torch.Tensor, draws: torch.Tensor) -> List[torch.Tensor]:
        """Folded encoder once; main decoder on the clean features, auxiliary decoder a on its perturbed copy of them
        (the reference's eval-mode forward, UAPS_unet.py:224-233); the draws are read from the device tensor ``draws``."""
        enc, dec, out, _ = self._inference_plan()
        feats = self._encode_folded(x, enc)
        keys, uth = draws[0], draws[1]

        def perturb(i, f, outputs):
            return P.perturb3_nhwc(f.permute(0, 3, 1, 2), outputs=outputs, seed_dev=keys[i].data_ptr(),
                                   u_dev=uth[i].data_ptr())

        live = tuple(a <= self.n_aux for a in (1, 2, 3))
        per_level = [perturb(lvl, f, live) for lvl, f in enumerate(feats)]
        logits = [self._decode_folded(feats, dec, out)]
        for a in range(1, self.n_aux + 1):
            kind = _AUX_KINDS[(a - 1) % 3]
            if a <= 3:
                pf = [t[a - 1] for t in per_level]
            else:                                             # a fresh draw of the family, as _forward16 does
                sel = tuple(k == kind for k in _AUX_KINDS)
                pf = [perturb(5 * (a - 3) + lvl, f, sel)[_AUX_KINDS.index(kind)] for lvl, f in enumerate(feats)]
            logits.append(self._decode_folded([t.permute(0, 2, 3, 1) for t in pf], *self._aux_plan(a)))
        return logits

    def _check_ensemble_input(self, x: torch.Tensor) -> None:
        if self.n_aux == 0:
            raise ValueError("predict_uncertainty needs at least one auxiliary decoder (n_aux >= 1)")
        _check_hw(x)

    @torch.no_grad()
    def predict_uncertainty(self, x: torch.Tensor, *, seed: Optional[int] = None, return_probs: bool = False):
        """Ensemble inference (UAPS-Testing.ipynb cell 11; DESIGN.md f5): every decoder's logits, then
        ``ensemble.ensemble_uncertainty`` -- ``(labels uint8 [B,H,W], uncertainty fp32 [B,H,W], image_uncertainty fp32 [B],
        mean_prob fp32 [B,C,H,W] | None)``: the argmax of the decoders' mean softmax, the mean KL divergence of each
        decoder from that mean per pixel (0 where they agree) and its per-image mean.

        As in the reference's eval-mode forward, the main decoder sees the clean encoder features and auxiliary decoder a
        a perturbed copy (FeatureNoise, Dropout(0.5), FeatureDropout for a = 1, 2, 3; a = 4, 5 a fresh draw of the first
        two families); the encoder's own dropout is off.

        bf16 path in eval mode: the folded encoder runs once, every decoder through BN-folded packed convs, the
        perturbations are the Philox kernels of training, and the head is one ``uaps_ensemble_head`` launch.  The random
        draws are n = 5 * (1 + max(0, n_aux - 3)) (Philox key, FeatureDropout u) pairs, one per perturbation launch, in
        the order: levels 0-4 of the shared launch for decoders 1-3, then levels 0-4 for decoder 4, then for decoder 5.
        Launch i takes key_i = rng.integers(0, 2**63 - 1), then u_i = rng.uniform(0.7, 0.9) (rounded to fp32), where rng
        is ``numpy.random.default_rng(seed)`` for an int ``seed`` and ``uaps_b200.perturb.generator`` for ``seed=None``.
        In training mode and on the fp32 path it runs ``forward(x)`` (whose draws come from the generator; ``seed`` is
        not used there) and the same head."""
        self._check_ensemble_input(x)
        from .ensemble import ensemble_uncertainty
        if self.compute == "bf16" and not self.training:
            draws = torch.from_numpy(self._ensemble_draws(seed)).to(x.device)       # one host-to-device copy
            logits = self._ensemble_logits16(x, draws)
        else:
            logits = self.forward(x)
        return ensemble_uncertainty(logits, return_probs=return_probs)

    @torch.no_grad()
    def predict_uncertainty_graphed(self, x: torch.Tensor, *, seed: Optional[int] = None):
        """``predict_uncertainty`` replayed from a CUDA graph (bf16 path, eval mode), one graph per input shape, as
        ``predict_graphed``.  The draws live in a static device buffer that receives fresh draws (from ``seed`` as
        ``predict_uncertainty`` derives them) before every replay.  The returned tensors are the graph's static output
        buffers: the next call with the same shape overwrites them."""
        if self.compute != "bf16" or self.training:
            return self.predict_uncertainty(x, seed=seed)
        self._check_ensemble_input(x)
        from .ensemble import ensemble_uncertainty
        key = ("uncertainty", tuple(x.shape), x.device.index)
        cache = self.__dict__.setdefault("_graphs", {})
        entry = cache.get(key)
        host_draws = torch.from_numpy(self._ensemble_draws(seed))
        if entry is None or entry[4] is not self._inference_plan():
            static_in = torch.empty_like(x, dtype=torch.float32)
            static_in.copy_(x)
            static_draws = host_draws.to(x.device)
            run = lambda: ensemble_uncertainty(self._ensemble_logits16(static_in, static_draws))
            side = torch.cuda.Stream(device=x.device)
            side.wait_stream(torch.cuda.current_stream(x.device))
            with torch.cuda.stream(side):                       # warm-up off the capture: lazy inits, plans, allocator
                for _ in range(2):
                    run()
            torch.cuda.current_stream(x.device).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_out = run()
            entry = (graph, static_in, static_draws, static_out, self._inference_plan())
            cache[key] = entry
        graph, static_in, static_draws, static_out, _ = entry
        static_in.copy_(x)
        static_draws.copy_(host_draws)
        graph.replay()
        return static_out

    def decoders(self) -> List[nn.Module]:
        return [self.main_decoder] + [self.get_submodule(f"aux_decoder{a}") for a in range(1, self.n_aux + 1)]

    # ---- forward ----------------------------------------------------------------------------
    def forward(self, x: torch.Tensor, rand: Optional[Dict[str, list]] = None):
        """UNet_UAPS.forward (:224-233).  ``rand`` optionally injects every random draw:
        {"enc_keep": 5 masks, "noise": 5 tensors [C_l,H_l,W_l], "aux2_keep": 5 masks, "u": 5 floats}."""
        _check_hw(x)
        if self.compute == "bf16":
            return self._forward16(x, rand)
        feats = self.encode(x, None if rand is None else rand["enc_keep"])
        outs = [self.decode(feats, self.main_decoder)]
        if self.n_aux == 0:
            return outs[0]
        per_kind: Dict[str, List[torch.Tensor]] = {k: [] for k in _AUX_KINDS}
        for lvl, f in enumerate(feats):
            kw = {} if rand is None else {"noise": rand["noise"][lvl], "keep": rand["aux2_keep"][lvl], "u": rand["u"][lvl]}
            yn, yd, yf = P.perturb3(f, **kw)
            per_kind["noise"].append(yn); per_kind["dropout"].append(yd); per_kind["fdrop"].append(yf)
        for a in range(1, self.n_aux + 1):
            kind = _AUX_KINDS[(a - 1) % 3]
            if a <= 3:
                pf = per_kind[kind]
            elif kind == "noise":                              # aux4+: a fresh draw of the same perturbation family
                pf = [P.FeatureNoise()(f) for f in feats]
            elif kind == "dropout":
                pf = [P.Dropout(f) for f in feats]
            else:
                pf = [P.FeatureDropout(f) for f in feats]
            outs.append(self.decode(pf, self.get_submodule(f"aux_decoder{a}")))
        return tuple(outs)


def load_reference_state_dict(model: nn.Module, state_dict: Dict[str, torch.Tensor], strict: bool = True):
    """Load a reference checkpoint's ``state_dict`` (UAPS_train.py:443-450), with or without the
    ``module.`` prefix that ``nn.DataParallel`` (UAPS_model.py:13) puts on every key."""
    cleaned = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in state_dict.items()}
    return model.load_state_dict(cleaned, strict=strict)


def inference_params(model_or_state_dict, *, ensemble: bool = False) -> torch.Tensor:
    """The parameter blob of the C inference entry points (``uaps_unet_infer_prepare``, include/uaps_b200.h): the
    ``encoder.*`` and ``main_decoder.*`` tensors of the state_dict in state_dict order, without ``num_batches_tracked``,
    flattened into one contiguous fp32 tensor on the tensors' device.  Takes a model or a state_dict, with or without the
    ``module.`` prefix of a reference checkpoint.

    ``ensemble=True``: the blob of ``uaps_unet_ensemble_prepare`` -- the same, followed by every ``aux_decoderN.*``
    tensor (N = 1 .. n_aux, state_dict order).  n_aux is read from the keys; it must be 1..5 with no gap."""
    sd = model_or_state_dict.state_dict() if isinstance(model_or_state_dict, nn.Module) else model_or_state_dict
    sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in sd.items()}
    prefixes = ("encoder.", "main_decoder.")
    if ensemble:
        found = sorted({int(m.group(1)) for k in sd if (m := re.match(r"aux_decoder(\d+)\.", k))})
        n_aux = len(found)
        if found != list(range(1, n_aux + 1)) or not 1 <= n_aux <= 5:
            raise ValueError(f"the ensemble blob needs auxiliary decoders 1..n_aux with n_aux in 1..5; the state_dict has "
                             f"{['aux_decoder%d' % a for a in found] or 'none'}")
        prefixes += tuple(f"aux_decoder{a}." for a in found)
    parts = [v.detach().reshape(-1).float() for k, v in sd.items()
             if k.startswith(prefixes) and not k.endswith("num_batches_tracked")]
    try:
        in_chns = sd["encoder.in_conv.conv_conv.0.weight"].shape[1]
        C = sd["main_decoder.out_conv.weight"].shape[0]
    except KeyError as e:
        raise ValueError(f"not a UNet_UAPS state_dict: {e} is missing") from None
    from . import _lib as L
    blob = torch.cat(parts)
    want = L.lib().uaps_unet_ensemble_params_count(in_chns, C, n_aux) if ensemble else L.lib().uaps_unet_params_count(in_chns, C)
    if blob.numel() != want:
        what = f"{in_chns} input channels, {C} classes" + (f", {n_aux} auxiliary decoders" if ensemble else "")
        raise ValueError(f"parameter blob of {blob.numel()} values, the network ({what}) needs {want}")
    return blob


def save_checkpoint(path: str, model: nn.Module, optimizer, epoch: int, best_dice: float, data_parallel_keys: bool = True):
    """The reference's checkpoint dict (UAPS_train.py:443-450): {"epoch", "best_dice_1", "state_dict", "optimizer"},
    with the ``module.`` key prefix its DataParallel wrapper produces, so the reference's notebooks can load it."""
    sd = model.state_dict()
    if data_parallel_keys:
        sd = {"module." + k: v for k, v in sd.items()}
    torch.save({"epoch": epoch, "best_dice_1": best_dice, "state_dict": sd, "optimizer": optimizer.state_dict()}, path)


def load_checkpoint(path: str, model: nn.Module, optimizer=None, map_location=None):
    ck = torch.load(path, map_location=map_location)
    load_reference_state_dict(model, ck["state_dict"])
    if optimizer is not None and "optimizer" in ck:
        optimizer.load_state_dict(ck["optimizer"])
    return ck.get("epoch"), ck.get("best_dice_1")


def net_factory(net_type: str = "unet_uaps", in_chns: int = 3, class_num: int = 4, compute: str = "bf16"):
    """utilities/UAPS_net_factory.py:5-13: the model on CUDA, or None for an unknown type.
    The model it returns runs the hand-written sm_100a kernels (``compute="bf16"``); pass ``compute="reference"`` for the
    fp32 torch/cuDNN path that exists for parity runs."""
    if net_type == "unet_uaps":
        return UNet_UAPS(in_chns=in_chns, class_num=class_num, compute=compute).cuda()
    if net_type == "unet":
        return UNet_UAPS(in_chns=in_chns, class_num=class_num, n_aux=0, compute=compute).cuda()
    return None
