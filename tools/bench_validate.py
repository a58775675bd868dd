#!/usr/bin/env python
"""Per-epoch validation on one B200 (DESIGN.md f6): prints one JSON line and, with --out, writes it to a file.

    python tools/bench_validate.py [--out profiles/f6_validate_b200.json] [--reps 10] [--rounds 5]

Per validation batch, at the three data-set shapes (NEU 64x256x256 C4, DAGM 32x512x512 C2 with one input channel,
KolektorSDD2 32x240x640 C2), device-resident inputs, CUDA events around `reps` batches:
  (a) graph     : Validator.update (folded main decoder + validation head, replayed from a CUDA graph);
  (b) predict   : predict + ce_loss + MetricAccumulator.update (the pieces a user could assemble before);
  (c) drop-in   : eval-mode model(x)[0] + ce_loss + MetricAccumulator.update (what a drop-in user runs today).
Head alone: uaps_val_counts + uaps_val_fold against uaps_confusion on the same logits.  Each timed call reads one of
several copies of logits + labels whose total exceeds the 126 MB L2 twice, so every call reads them from HBM.
Algorithmic bytes per pixel: 4C (logits) + 8 (int64 label).  All paths are interleaved round by round; medians with the
spread are reported.
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

CASES = [("neu_64x256x256_C4", 3, 4, 64, 256, 256), ("dagm_32x512x512_C2_in1", 1, 2, 32, 512, 512),
         ("kosdd2_32x240x640_C2", 3, 2, 32, 240, 640)]
L2_BYTES = 126 << 20


def bench_case(name, cin, C, B, H, W, reps, rounds):
    from uaps_b200 import _lib as L
    from uaps_b200.losses import ce_loss
    from uaps_b200.metrics import MetricAccumulator, confusion
    from uaps_b200.unet import UNet_UAPS
    from uaps_b200.validate import Validator
    lib = L.lib()
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = UNet_UAPS(cin, C).to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(B, cin, H, W, generator=g, device=dev)
    y = torch.randint(0, C, (B, H, W), generator=g, device=dev)
    val = Validator(model, max_batches=reps + 4)
    acc = MetricAccumulator(dev)

    def graph():
        val.update(x, y)

    def predict():
        logits = model.predict(x)
        ce_loss(logits, y)
        acc.update(logits, y)

    def dropin():
        with torch.no_grad():
            logits = model(x)[0]
        ce_loss(logits, y)
        acc.update(logits, y)

    # head alone, on logits of this model and shape; copies rotate so that no call finds its inputs in L2
    HW = H * W
    per_call = B * HW * (4 * C + 8)
    n_copies = max(2, -(-2 * L2_BYTES // per_call))
    base = model.predict(x)
    zs = [base + 1e-3 * i for i in range(n_copies)]
    ys = [y.roll(i, 0).contiguous() for i in range(n_copies)]
    ws = torch.empty(lib.uaps_val_workspace_bytes(C, B, HW), dtype=torch.uint8, device=dev)
    table = torch.zeros(reps * n_copies + 4, C * C + 3, dtype=torch.float64, device=dev)
    state = torch.zeros(3, dtype=torch.int32, device=dev)
    conf = torch.zeros(C, C, dtype=torch.int64, device=dev)
    it = {"head": 0, "conf": 0}

    def head():
        i = it["head"] = (it["head"] + 1) % n_copies
        st = L.stream_ptr()
        L.check(lib.uaps_val_counts(zs[i].data_ptr(), ys[i].data_ptr(), B, C, HW, ws.data_ptr(), ws.numel(), st), "counts")
        L.check(lib.uaps_val_fold(ws.data_ptr(), ws.numel(), B, C, HW, table.data_ptr(), table.shape[0], state.data_ptr(),
                                  st), "fold")

    def conf_only():
        i = it["conf"] = (it["conf"] + 1) % n_copies
        confusion(zs[i], ys[i], out=conf)

    val.begin()
    for fn in (graph, graph, graph, predict, dropin):         # eager, capture, replay; lazy initialisation of the others
        fn()
    samples = {k: [] for k in ("graph", "predict", "dropin", "head", "confusion")}
    for _ in range(rounds):
        val.begin()
        state.zero_()
        samples["graph"].append(event_ms(graph, reps))
        samples["predict"].append(event_ms(predict, reps))
        samples["dropin"].append(event_ms(dropin, reps))
        samples["head"].append(event_ms(head, reps * n_copies) * 1e3)
        samples["confusion"].append(event_ms(conf_only, reps * n_copies) * 1e3)
    res = val.result()
    out = {"shape": [B, cin, H, W], "classes": C, "captures": val.captures,
           "ms_per_batch": {k: summary(samples[k]) for k in ("graph", "predict", "dropin")},
           "us_head": {"val_counts+fold": summary(samples["head"]), "uaps_confusion": summary(samples["confusion"])},
           "head_bytes_per_call": per_call, "head_gbs": per_call / (statistics.median(samples["head"]) * 1e-6) / 1e9,
           "confusion_gbs": B * HW * (4 * C + 8) / (statistics.median(samples["confusion"]) * 1e-6) / 1e9,
           "input_copies": n_copies, "val_result": res}
    med = {k: statistics.median(samples[k]) for k in samples}
    out["speedup_vs_predict"] = med["predict"] / med["graph"]
    out["speedup_vs_dropin"] = med["dropin"] / med["graph"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_validate.py measures the B200: no CUDA device found")
    res = {"bench": "f6_validate", "gpu": gpu_info(), "reps": a.reps, "rounds": a.rounds,
           "cases": {name: bench_case(name, *rest, reps=a.reps, rounds=a.rounds) for name, *rest in CASES}}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
