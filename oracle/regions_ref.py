"""Host reference of the defect regions (uaps_regions, DESIGN.md f10) with numpy / scipy -- test infrastructure only.

For every nonzero class c, ``scipy.ndimage.label(labels == c, structure=np.ones((3, 3)))`` gives the 8-connected
components of that class.  They are renumbered 1..n per image by their smallest raster index y * W + x; area comes from
``bincount``, the half-open boxes from ``find_objects`` and the uncertainty sums from an fp64 ``bincount`` with weights,
so ``unc_mean`` is the fp64 mean rounded once to fp32.
"""
from __future__ import annotations

import numpy as np
from scipy import ndimage

_EIGHT = np.ones((3, 3), dtype=bool)


def regions_ref_image(labels: np.ndarray, uncertainty: np.ndarray | None = None):
    """labels uint8 [H, W] (uncertainty fp32 [H, W] or None) -> dict of regions int32 [H, W] and per region (id order)
    cls, area, bbox [n, 4] = (y0, x0, y1, x1), unc_mean fp32."""
    labels = np.asarray(labels)
    H, W = labels.shape
    comp = np.zeros((H, W), dtype=np.int64)
    n = 0
    for c in np.unique(labels):
        if c == 0:
            continue
        lab, k = ndimage.label(labels == c, structure=_EIGHT)
        comp[lab > 0] = lab[lab > 0] + n
        n += k
    flat = comp.reshape(-1)
    first = np.full(n + 1, H * W, dtype=np.int64)               # smallest raster index of every component
    np.minimum.at(first, flat, np.arange(H * W))
    order = np.argsort(first[1:], kind="stable")               # components in raster order of their first pixel
    new_id = np.zeros(n + 1, dtype=np.int64)
    new_id[1 + order] = np.arange(1, n + 1)
    regions = new_id[comp].astype(np.int32)
    rflat = regions.reshape(-1)
    area = np.bincount(rflat, minlength=n + 1)[1:].astype(np.int32)
    bbox = np.zeros((n, 4), dtype=np.int32)
    for i, sl in enumerate(ndimage.find_objects(regions)):
        bbox[i] = (sl[0].start, sl[1].start, sl[0].stop, sl[1].stop)
    firsts = np.sort(first[1:])
    cls = labels.reshape(-1)[firsts].astype(np.int32) if n else np.zeros(0, dtype=np.int32)
    if uncertainty is None:
        unc_mean = np.zeros(n, dtype=np.float32)
    else:
        sums = np.bincount(rflat, weights=np.asarray(uncertainty, dtype=np.float64).reshape(-1), minlength=n + 1)[1:]
        unc_mean = (sums / np.maximum(area, 1)).astype(np.float32)
    return {"regions": regions, "count": n, "cls": cls, "area": area, "bbox": bbox, "unc_mean": unc_mean}


def regions_ref(labels: np.ndarray, uncertainty: np.ndarray | None = None):
    """Batched: labels uint8 [B, H, W] -> list of per-image dicts (regions_ref_image)."""
    return [regions_ref_image(labels[b], None if uncertainty is None else uncertainty[b]) for b in range(labels.shape[0])]
