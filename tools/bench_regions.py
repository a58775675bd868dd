#!/usr/bin/env python
"""Defect regions (DESIGN.md f10) on one B200: prints one JSON line and, with --out, writes it to a file.

    python tools/bench_regions.py [--out profiles/f10_regions_b200.json] [--reps 50] [--rounds 5] [--host-reps 3]

Per batch shape (64x256x256, 32x512x512, 32x240x640) and label map (smooth blobs, density-0.4 noise of 3 classes,
one region covering every image, a one-pixel serpentine through every image):
  (a) uaps_regions with the uncertainty map and max_regions = 256: CUDA events around `reps` calls, the maps
      interleaved round by round, median and spread over `rounds`;
  (b) UNet_UAPS(3, 4, n_aux=3).predict_uncertainty_graphed on a batch of that shape, the ensemble forward that produces
      the maps, CUDA events the same way;
  (c) the host path a caller has without (a): copy labels and uncertainty to the host, then scipy.ndimage.label per class
      with the stats (the oracle, oracle/regions_ref.py), on one thread and on a pool of min(host cores, 64) processes;
      wall clock, median of `host_reps`.
The device results are checked against the oracle on every map before any timing.  A torch.profiler pass of its own
(the blob map at 64x256x256) gives the time of each kernel of (a).
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import json
import multiprocessing as mp
import os
import statistics
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_ensemble import event_ms, gpu_info, summary  # noqa: E402
from oracle.regions_ref import regions_ref_image  # noqa: E402

SHAPES = ((64, 256, 256), (32, 512, 512), (32, 240, 640))
MAPS = ("blob", "noise0.4", "full", "serpentine")
MAX_REGIONS = 256


def make_map(kind, B, H, W, seed=0):
    from scipy import ndimage
    rng = np.random.default_rng(seed)
    if kind == "blob":                  # thresholded Gaussian-filtered noise, 3 defect classes
        out = np.zeros((B, H, W), dtype=np.uint8)
        for b in range(B):
            for c in (1, 2, 3):
                f = ndimage.gaussian_filter(rng.standard_normal((H, W)).astype(np.float32), 6.0)
                out[b][f > 0.9 * f.std()] = c
        return out
    if kind == "noise0.4":
        fg = rng.random((B, H, W)) < 0.4
        return np.where(fg, rng.integers(1, 4, size=(B, H, W)), 0).astype(np.uint8)
    if kind == "full":
        return np.ones((B, H, W), dtype=np.uint8)
    m = np.zeros((H, W), dtype=np.uint8)
    m[0::2] = 1
    for y in range(1, H, 2):
        m[y, W - 1 if (y // 2) % 2 == 0 else 0] = 1
    return np.broadcast_to(m, (B, H, W)).copy()


def host_one(labels, unc):
    return [regions_ref_image(labels[b], unc[b])["count"] for b in range(labels.shape[0])]


def host_path(labels_d, unc_d, pool, workers):
    """Copy to the host, then label + stats per image: one thread, and split over the pool's processes."""
    t0 = time.perf_counter()
    labels, unc = labels_d.cpu().numpy(), unc_d.cpu().numpy()
    t1 = time.perf_counter()
    host_one(labels, unc)
    t2 = time.perf_counter()
    parts = np.array_split(np.arange(labels.shape[0]), workers)
    list(pool.map(host_one, [labels[p] for p in parts if p.size], [unc[p] for p in parts if p.size]))
    t3 = time.perf_counter()
    return (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--host-reps", type=int, default=3)
    a = ap.parse_args()
    # the host pool is forked before CUDA is initialised; more processes than images per batch would idle
    cores = os.cpu_count() or 1
    workers = min(cores, max(s[0] for s in SHAPES))
    pool = cf.ProcessPoolExecutor(max_workers=workers, mp_context=mp.get_context("fork"))
    list(pool.map(host_one, [np.zeros((1, 8, 8), np.uint8)] * workers, [np.zeros((1, 8, 8), np.float32)] * workers))
    if not torch.cuda.is_available():
        raise SystemExit("bench_regions.py measures the B200: no CUDA device found")
    from uaps_b200 import _lib as L
    from uaps_b200.unet import UNet_UAPS
    lib = L.lib()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = UNet_UAPS(3, 4, n_aux=3).to(dev).eval()

    results = {}
    for B, H, W in SHAPES:
        shape = f"{B}x{H}x{W}"
        g = torch.Generator(device=dev).manual_seed(1)
        unc = torch.rand((B, H, W), generator=g, device=dev)
        regions = torch.empty((B, H, W), dtype=torch.int32, device=dev)
        count = torch.empty(B, dtype=torch.int32, device=dev)
        stats = torch.empty((B, MAX_REGIONS, 8), dtype=torch.int32, device=dev)
        nbytes = lib.uaps_regions_workspace_bytes(B, H, W, MAX_REGIONS)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        calls = {}
        for kind in MAPS:
            labels = torch.from_numpy(make_map(kind, B, H, W)).to(dev)
            args = (labels.data_ptr(), unc.data_ptr(), B, H, W, regions.data_ptr(), count.data_ptr(), stats.data_ptr(),
                    MAX_REGIONS, ws.data_ptr(), nbytes)
            call = (lambda args=args: L.check(lib.uaps_regions(*args, L.stream_ptr()), "uaps_regions"))
            call()
            torch.cuda.synchronize()
            ref = [regions_ref_image(m, u) for m, u in zip(labels.cpu().numpy(), unc.cpu().numpy())]
            assert np.array_equal(regions.cpu().numpy(), np.stack([r["regions"] for r in ref])), (shape, kind)
            assert count.cpu().tolist() == [r["count"] for r in ref], (shape, kind)
            calls[kind] = (call, labels)
        x = torch.randn(B, 3, H, W, generator=g, device=dev)
        fwd = lambda: model.predict_uncertainty_graphed(x, seed=3)       # noqa: E731
        for _ in range(3):
            fwd()
        samples = {k: [] for k in MAPS}
        samples["predict_uncertainty_graphed"] = []
        for r in range(a.rounds):
            order = list(samples) if r % 2 == 0 else list(reversed(list(samples)))
            for k in order:
                fn = fwd if k == "predict_uncertainty_graphed" else calls[k][0]
                samples[k].append(event_ms(fn, a.reps if fn is not fwd else max(1, a.reps // 10)))
        host = {}
        for k in MAPS:
            runs = [host_path(calls[k][1], unc, pool, workers) for _ in range(a.host_reps)]
            host[k] = {"d2h_ms": statistics.median(r[0] for r in runs),
                       "scipy_1thread_ms": statistics.median(r[1] for r in runs),
                       f"scipy_{workers}proc_ms": statistics.median(r[2] for r in runs)}
        fwd_ms = statistics.median(samples["predict_uncertainty_graphed"])
        results[shape] = {
            "uaps_regions_ms": {k: summary(samples[k]) for k in MAPS},
            "predict_uncertainty_graphed_ms": summary(samples["predict_uncertainty_graphed"]),
            "regions_over_forward": {k: statistics.median(samples[k]) / fwd_ms for k in MAPS},
            "host_path": host,
        }
        del calls, regions, stats, ws, unc, x
        torch.cuda.empty_cache()
    pool.shutdown()

    # per-kernel times of the blob map at the first shape, in a run of their own
    from torch.profiler import ProfilerActivity, profile
    B, H, W = SHAPES[0]
    labels = torch.from_numpy(make_map("blob", B, H, W)).to(dev)
    unc = torch.rand((B, H, W), device=dev)
    regions = torch.empty((B, H, W), dtype=torch.int32, device=dev)
    count = torch.empty(B, dtype=torch.int32, device=dev)
    stats = torch.empty((B, MAX_REGIONS, 8), dtype=torch.int32, device=dev)
    nbytes = lib.uaps_regions_workspace_bytes(B, H, W, MAX_REGIONS)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    args = (labels.data_ptr(), unc.data_ptr(), B, H, W, regions.data_ptr(), count.data_ptr(), stats.data_ptr(),
            MAX_REGIONS, ws.data_ptr(), nbytes)
    for _ in range(5):
        L.check(lib.uaps_regions(*args, L.stream_ptr()), "uaps_regions")
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            L.check(lib.uaps_regions(*args, L.stream_ptr()), "uaps_regions")
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        if "regions_" in ev.key:
            name = ev.key.split("regions_", 1)[1].split("_kernel")[0]
            kernels[name] = round(ev.device_time_total / 1e3 / ev.count, 5)

    out = {"bench": "f10_regions", "gpu": gpu_info(), "host_cores": cores, "host_pool_processes": workers,
           "workload": f"uaps_regions with an uncertainty map, max_regions={MAX_REGIONS}; maps {list(MAPS)}; "
                       "predict_uncertainty_graphed: UNet_UAPS(3, 4, n_aux=3), bf16, eval",
           "reps_per_sample": a.reps, "rounds": a.rounds, "shapes": results,
           "kernel_ms_blob_64x256x256": kernels}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
