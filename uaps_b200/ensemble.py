"""Ensemble inference over UAPS's decoders: label map and uncertainty maps from K decoders' logits.

The reference draws its test-time uncertainty from the disagreement between the main and the auxiliary decoders
(UAPS-Testing.ipynb cell 11) with the expressions of its uncertainty loss (UAPS_train.py:186-189, 223-243).
``ensemble_uncertainty`` computes, in one kernel (``uaps_ensemble_head``) plus a per-image fold:

* ``labels``            uint8 [B,H,W]: argmax_c q with q = (p_0 + ... + p_{K-1}) / K, p_k = softmax(z_k) --
  bit-exact with ``torch.argmax(q, 1)`` (lowest index on ties);
* ``uncertainty``       fp32 [B,H,W]: (1/K) sum_k sum_c KLDiv(log_softmax(z_k), q), the per-pixel term of the uncertainty
  loss -- 0 where the decoders agree;
* ``image_uncertainty`` fp32 [B]: its mean over each image's pixels, summed in fp64 in a fixed order (bitwise
  reproducible), e.g. to route doubtful parts to a human;
* ``mean_prob``         fp32 [B,C,H,W]: q, only with ``return_probs=True``.

Inference only: there is no backward.  CUDA tensors only; no fallback.
"""
from __future__ import annotations

from typing import NamedTuple, Optional, Sequence

import torch

from . import _lib as L
from .losses import _prep_logits


class EnsembleOutput(NamedTuple):
    labels: torch.Tensor
    uncertainty: torch.Tensor
    image_uncertainty: torch.Tensor
    mean_prob: Optional[torch.Tensor]


@torch.no_grad()
def ensemble_uncertainty(logits: Sequence[torch.Tensor], *, return_probs: bool = False) -> EnsembleOutput:
    """logits: K (1..6) fp32 CUDA tensors [B, C, H, W] of the same shape, C in 2..8 (main decoder first, as
    ``UNet_UAPS.forward`` returns them).  Returns ``EnsembleOutput(labels, uncertainty, image_uncertainty, mean_prob)``."""
    zs, B, C, H, W = _prep_logits(logits)
    K, HW = len(zs), H * W
    dev = zs[0].device
    lib = L.lib()
    with L.on_device(dev):
        labels = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        unc = torch.empty((B, H, W), dtype=torch.float32, device=dev)
        img = torch.empty(B, dtype=torch.float32, device=dev)
        q = torch.empty((B, C, H, W), dtype=torch.float32, device=dev) if return_probs else None
        nbytes = lib.uaps_ensemble_workspace_bytes(K, C, B, HW)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)      # per-chunk partial sums, all written before read
        L.check(lib.uaps_ensemble_head(L.ptr_array(zs), K, B, C, HW, labels.data_ptr(), unc.data_ptr(), img.data_ptr(),
                                       None if q is None else q.data_ptr(), ws.data_ptr(), nbytes, L.stream_ptr()),
                "uaps_ensemble_head")
    return EnsembleOutput(labels, unc, img, q)
