#!/usr/bin/env python
"""Ensemble inference on one B200 (DESIGN.md f5): prints one JSON line and, with --out, writes it to a file.

    python tools/bench_ensemble.py [--out profiles/f5_ensemble.json] [--reps 50] [--rounds 5]

head : uaps_ensemble_head (+ the per-image fold) on the DAGM / NEU / KolektorSDD2 shapes, C-ABI calls with preallocated
       outputs, timed with CUDA events; in the same run and on the same logits, loss pass 1 (uaps_loss_pass1 without the
       optional per-pixel outputs) -- the same per-pixel softmax / KL work plus the loss sums.  The logits of every
       shape (196..268 MB) exceed the 126 MB L2, so every call reads them from HBM.  Algorithmic bytes per pixel:
       4KC + 1 + 4 (labels, uncertainty), + 4C with the mean prediction; against the measured 6538.9 GB/s copy rate.
e2e  : host images in, uint8 label map + fp32 uncertainty map out (the method of bench.py's inference block), at B = 64
       and batch 1 (plain launches and CUDA graph), beside predict (main decoder only) and the incumbent a user writes
       without this path: eval-mode forward() and the oracle's torch expressions for the mean prediction and KL maps.
Head timings and the three e2e paths are interleaved round by round; medians are reported with the spread.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_GBS = 6538.9                 # measured HBM copy rate of the project's B200 (BASELINE.md)
PUBLISHED_MS = {"main+1": 25.72, "main+2": 26.84, "main+3": 29.47, "main+4": 33.79}   # paper's decoder-effect figure
HEAD_CASES = [("neu_64x256x256_K4C4", 4, 4, 64, 256, 256), ("dagm_32x512x512_K4C2", 4, 2, 32, 512, 512),
              ("kosdd2_32x240x640_K5C2", 5, 2, 32, 240, 640)]


def gpu_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else r.stderr.strip()
    except Exception as e:              # noqa: BLE001 -- recorded, not fatal
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def event_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def summary(samples):
    return {"median": statistics.median(samples), "min": min(samples), "max": max(samples)}


def head_bench(reps, rounds):
    from uaps_b200 import _lib as L
    lib = L.lib()
    dev = torch.device("cuda:0")
    out = {}
    for name, K, C, B, H, W in HEAD_CASES:
        HW = H * W
        g = torch.Generator(device=dev).manual_seed(1)
        z = [torch.randn(B, C, H, W, device=dev, generator=g) * 2 for _ in range(K)]
        zp = L.ptr_array(z)
        labels = torch.empty(B, HW, dtype=torch.uint8, device=dev)
        unc = torch.empty(B, HW, device=dev)
        img = torch.empty(B, device=dev)
        q = torch.empty(B, C, HW, device=dev)
        nws = lib.uaps_ensemble_workspace_bytes(K, C, B, HW)
        ws = torch.empty(nws, dtype=torch.uint8, device=dev)
        lws = torch.zeros(lib.uaps_loss_workspace_bytes(K, C), dtype=torch.uint8, device=dev)
        sums = torch.empty(lib.uaps_loss_sums_count(K, C), dtype=torch.float64, device=dev)
        mix_w = L.float_array([1.0 / K] * K)
        st = L.stream_ptr()

        def head(probs=False):
            L.check(lib.uaps_ensemble_head(zp, K, B, C, HW, labels.data_ptr(), unc.data_ptr(), img.data_ptr(),
                                           q.data_ptr() if probs else None, ws.data_ptr(), nws, st), "uaps_ensemble_head")

        def pass1():
            L.check(lib.uaps_loss_pass1(zp, K, B, C, HW, mix_w, None, lws.data_ptr(), sums.data_ptr(), None, None, 0, st),
                    "uaps_loss_pass1")

        for f in (head, lambda: head(True), pass1):
            for _ in range(3):
                f()
        torch.cuda.synchronize()
        t_head, t_probs, t_p1 = [], [], []
        for _ in range(rounds):
            t_head.append(event_ms(head, reps))
            t_p1.append(event_ms(pass1, reps))
            t_probs.append(event_ms(lambda: head(True), reps))
        npx = B * HW
        bytes_head = npx * (4 * K * C + 5)
        bytes_probs = bytes_head + npx * 4 * C
        mh, mp, m1 = (statistics.median(t) for t in (t_head, t_probs, t_p1))
        out[name] = {
            "K": K, "C": C, "B": B, "H": H, "W": W,
            "head_us": {k: v * 1e3 for k, v in summary(t_head).items()},
            "head_with_probs_us": {k: v * 1e3 for k, v in summary(t_probs).items()},
            "loss_pass1_us": {k: v * 1e3 for k, v in summary(t_p1).items()},
            "head_gbs": bytes_head / (mh * 1e-3) / 1e9, "head_frac_hbm": bytes_head / (mh * 1e-3) / 1e9 / HBM_GBS,
            "head_with_probs_frac_hbm": bytes_probs / (mp * 1e-3) / 1e9 / HBM_GBS,
            "loss_pass1_frac_hbm": npx * 4 * K * C / (m1 * 1e-3) / 1e9 / HBM_GBS,
            "hbm_floor_us": bytes_head / (HBM_GBS * 1e9) * 1e6,
            "head_over_pass1": mh / m1,
            "head_not_slower_than_pass1": mh <= m1,
        }
        del z, q
        torch.cuda.empty_cache()
    return out


def e2e_bench(batch, steps, rounds):
    from oracle import uaps_loss_ref as R                                   # the incumbent's criteria modules
    from uaps_b200.unet import UNet_UAPS
    dev = torch.device("cuda:0")
    C, H, W = 4, 256, 256
    torch.manual_seed(1337)
    model = UNet_UAPS(3, C, n_aux=3, compute="bf16").to(dev).eval()
    K = 1 + model.n_aux

    def make(b):
        return (torch.randn(b, 3, H, W).pin_memory(), torch.empty((b, H, W), dtype=torch.uint8).pin_memory(),
                torch.empty((b, H, W), dtype=torch.float32).pin_memory())

    def ours(x_h, lab_h, unc_h, fn=model.predict_uncertainty):
        out = fn(x_h.to(dev, non_blocking=True))
        lab_h.copy_(out.labels, non_blocking=True)
        unc_h.copy_(out.uncertainty, non_blocking=True)

    def main_only(x_h, lab_h, unc_h, fn=model.predict):
        lab_h.copy_(fn(x_h.to(dev, non_blocking=True)).argmax(1).to(torch.uint8), non_blocking=True)

    @torch.no_grad()
    def incumbent(x_h, lab_h, unc_h):
        logits = model(x_h.to(dev, non_blocking=True))                     # eval-mode forward: BN through torch
        soft = [torch.softmax(z, dim=1) for z in logits]                    # UAPS_train.py:186-189
        acc = soft[0]
        for k in range(1, K):
            acc = acc + soft[k]
        preds = acc / K                                                     # :223
        var = [torch.sum(R._kl_none(R._log_sm(z), preds), dim=1) for z in logits]   # :226-236
        vsum = var[0]
        for k in range(1, K):
            vsum = vsum + var[k]
        lab_h.copy_(preds.argmax(1).to(torch.uint8), non_blocking=True)
        unc_h.copy_(vsum / K, non_blocking=True)

    bufs = make(batch)
    paths = {"predict_uncertainty": ours, "predict_main_only": main_only, "incumbent_forward_plus_torch_head": incumbent}
    for fn in paths.values():
        for _ in range(3):
            fn(*bufs)
    torch.cuda.synchronize()
    times = {k: [] for k in paths}
    for _ in range(rounds):
        for k, fn in paths.items():
            times[k].append(event_ms(lambda: fn(*bufs), steps))
    res = {k: {"ms_per_image": statistics.median(v) / batch, "ms_per_batch": summary(v)} for k, v in times.items()}

    b1 = make(1)
    lat = {}
    for name, fn in (("predict_uncertainty_launches", lambda *a: ours(*a)),
                     ("predict_uncertainty_cuda_graph", lambda *a: ours(*a, fn=model.predict_uncertainty_graphed)),
                     ("predict_launches", lambda *a: main_only(*a)),
                     ("predict_cuda_graph", lambda *a: main_only(*a, fn=model.predict_graphed)),
                     ("incumbent", incumbent)):
        def one():
            fn(*b1)
            torch.cuda.current_stream().synchronize()
        for _ in range(5):
            one()
        samples = []
        for _ in range(rounds):
            t0 = time.perf_counter()
            for _ in range(20):
                one()
            samples.append((time.perf_counter() - t0) / 20 * 1e3)
        lat[name] = summary(samples)
    ours_ms = res["predict_uncertainty"]["ms_per_image"]
    inc_ms = res["incumbent_forward_plus_torch_head"]["ms_per_image"]
    return {"config": f"UNet_UAPS n_aux=3 (K=4) 3x{H}x{W} C={C}, bf16 path, eval mode, host images in, "
                      "uint8 labels + fp32 uncertainty map out", "batch": batch, "timed_batches": steps,
            "throughput": res, "speedup_vs_incumbent": inc_ms / ours_ms, "faster_than_incumbent": ours_ms < inc_ms,
            "latency_ms_batch1": lat,
            "published_ms_per_image": PUBLISHED_MS,
            "published_source": "UAPS paper, decoder-effect figure (main + 1..4 auxiliary decoders; hardware not stated)"}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ensemble.py needs a CUDA device: uaps_b200 has no CPU path")
    res = {"bench": "ensemble_inference", "gpu": gpu_info(), "hbm_gbs_reference": HBM_GBS,
           "head": head_bench(args.reps, args.rounds), "e2e": e2e_bench(args.batch, args.steps, args.rounds)}
    res["gpu_after"] = gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
