"""Defect regions: connected components of a label map with per-region class, area, box and mean uncertainty.

An inspection line acts on defects rather than pixels: which connected patches of a defect class an image has, where
they are, how large they are and how sure the model is about each one.  ``defect_regions`` computes that on the device
from the outputs of ``UNet_UAPS.predict_uncertainty`` (or any uint8 label map), one ``uaps_regions`` call:

* a region is a maximal 8-connected set of pixels with the same nonzero label (class 0 is background; touching pixels
  of different classes belong to different regions);
* ids are 1..n per image in raster order of each region's first pixel, 0 for background -- independent of scheduling,
  so the map, counts and integer statistics are bitwise reproducible;
* ``unc_mean`` is the region's mean uncertainty (fp64 sum, rounded once to fp32), the per-defect form of
  ``image_uncertainty``: one doubtful speck no longer makes a confident scratch in the same image look doubtful.

    regions = defect_regions(*model.predict_uncertainty(x)[:2])

CUDA tensors only; no fallback.
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import torch

from . import _lib as L

_FIELDS = 8          # int32 words of UapsRegion: cls, area, y0, x0, y1, x1, unc_mean (fp32), reserved


class Regions(NamedTuple):
    regions: torch.Tensor      # int32 [B, H, W]: region id per pixel, 0 = background
    count: torch.Tensor        # int32 [B]: regions per image (also when it exceeds max_regions)
    cls: torch.Tensor          # int32 [B, max_regions]: class of region id i + 1; rows >= count are 0
    area: torch.Tensor         # int32 [B, max_regions]: pixels
    bbox: torch.Tensor         # int32 [B, max_regions, 4]: (y0, x0, y1, x1), half-open
    unc_mean: torch.Tensor     # fp32 [B, max_regions]: mean uncertainty (0 without an uncertainty map)


@torch.no_grad()
def defect_regions(labels: torch.Tensor, uncertainty: Optional[torch.Tensor] = None, *,
                   max_regions: int = 256) -> Regions:
    """labels: uint8 CUDA tensor [B, H, W] (pass ``labels.to(torch.uint8)`` for other integer maps); uncertainty:
    optional fp32 CUDA tensor of the same shape.  Returns ``Regions(regions, count, cls, area, bbox, unc_mean)``; the
    statistics are views of one [B, max_regions] table of ``UapsRegion`` rows, in id order, and cover the first
    ``max_regions`` regions of each image (the map numbers all of them)."""
    L.require_cuda(labels, uncertainty)
    if labels.dtype != torch.uint8:
        raise RuntimeError(f"labels must be uint8 (pass labels.to(torch.uint8)), got {labels.dtype}")
    if labels.dim() != 3:
        raise RuntimeError(f"labels must be [B, H, W], got shape {tuple(labels.shape)}")
    if max_regions < 0:
        raise RuntimeError(f"max_regions must be >= 0, got {max_regions}")
    B, H, W = labels.shape
    labels = labels.contiguous()
    if uncertainty is not None:
        if uncertainty.dtype != torch.float32 or uncertainty.shape != labels.shape:
            raise RuntimeError("uncertainty must be fp32 with the shape of labels")
        if uncertainty.device != labels.device:
            raise RuntimeError("labels and uncertainty must be on the same device")
        uncertainty = uncertainty.contiguous()
    dev = labels.device
    lib = L.lib()
    with L.on_device(dev):
        nbytes = lib.uaps_regions_workspace_bytes(B, H, W, max_regions)
        if nbytes == 0:
            raise RuntimeError(f"unsupported region shape B={B}, H={H}, W={W} (needs B <= 65535, H * W < 2^31)")
        regions = torch.empty((B, H, W), dtype=torch.int32, device=dev)
        count = torch.empty(B, dtype=torch.int32, device=dev)
        stats = torch.empty((B, max_regions, _FIELDS), dtype=torch.int32, device=dev)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)     # written before read inside the call
        L.check(lib.uaps_regions(labels.data_ptr(), None if uncertainty is None else uncertainty.data_ptr(), B, H, W,
                                 regions.data_ptr(), count.data_ptr(), stats.data_ptr() if max_regions > 0 else None,
                                 max_regions, ws.data_ptr(), nbytes, L.stream_ptr()),
                "uaps_regions")
    return Regions(regions, count, stats[..., 0], stats[..., 1], stats[..., 2:6], stats.view(torch.float32)[..., 6])
