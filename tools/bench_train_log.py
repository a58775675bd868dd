#!/usr/bin/env python
"""Cost of the training log (DESIGN.md f9) on one B200: prints one JSON line and, with --out, writes it to a file.

    python tools/bench_train_log.py [--out profiles/f9_train_log_b200.json] [--steps 20] [--rounds 5]

The captured UAPS iteration at the NEU shape (64 labeled + 64 unlabeled images of 3x256x256, C = 4, K = 4), device-resident
batches, from two trainers built from the same seed: one with the log off (UAPSConfig.train_log_rows = 0) and one with
it on.  CUDA events around `steps` iterations; the two trainers alternate round by round in the same process, and
medians with the spread are reported.  Before the timing, the two trainers' first iterations are compared, and the log's
epoch read-out is checked against the scalars the timed iterations returned.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_ensemble import event_ms, gpu_info, summary  # noqa: E402

B, CIN, H, W, C, K = 64, 3, 256, 256, 4, 4


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_log.py measures the B200: no CUDA device found")
    from uaps_b200.train import UAPSConfig, UAPSTrainer
    from uaps_b200.unet import UNet_UAPS
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    xl = torch.randn(B, CIN, H, W, generator=g, device=dev)
    xu = torch.randn(B, CIN, H, W, generator=g, device=dev)
    yl = torch.randint(0, C, (B, H, W), generator=g, device=dev)
    trainers = {}
    first = {}
    for name, rows in (("off", 0), ("on", a.steps + 8)):
        torch.manual_seed(1337)
        tr = UAPSTrainer(UNet_UAPS(CIN, C, n_aux=K - 1).to(dev), UAPSConfig(num_classes=C, train_log_rows=rows))
        first[name] = float(tr.step(xl, yl, xu)["loss"])
        for _ in range(3):                                   # second warm-up, capture, one replay
            tr.step(xl, yl, xu)
        trainers[name] = tr
    assert all(len(tr._graphs) == 1 for tr in trainers.values())
    on = trainers["on"]
    samples = {"off": [], "on": []}
    losses = []
    for r in range(a.rounds):
        for name in (("off", "on") if r % 2 == 0 else ("on", "off")):
            tr = trainers[name]
            if name == "on":
                tr.log_begin()
            samples[name].append(event_ms(lambda: tr.step(xl, yl, xu), a.steps))
    # the log of the last round against the scalars those iterations returned (one more epoch, not timed)
    on.log_begin()
    for _ in range(a.steps):
        losses.append(on.step(xl, yl, xu)["loss"].clone())
    res = on.log_result()
    mean_loss = torch.stack(losses).double().mean().item()
    med = {k: statistics.median(v) for k, v in samples.items()}
    out = {"bench": "f9_train_log", "gpu": gpu_info(),
           "workload": f"captured UAPSTrainer.step, NEU {B}+{B} x {CIN}x{H}x{W}, C={C}, K={K}, device-resident batches",
           "steps_per_sample": a.steps, "rounds": a.rounds,
           "ms_per_iter": {k: summary(v) for k, v in samples.items()},
           "overhead_pct": 100.0 * (med["on"] - med["off"]) / med["off"],
           "first_iteration_loss": first,
           "log_result": res, "log_loss_vs_returned_mean_rel": abs(res["loss"] - mean_loss) / abs(mean_loss)}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
