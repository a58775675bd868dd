#!/usr/bin/env python
"""Whole-network inference through the C ABI on one B200 (DESIGN.md f7): prints one JSON line and, with --out, writes it.

    python tools/bench_infer_c.py [--out profiles/f7_c_infer_b200.json] [--reps 50] [--rounds 5]

NEU shape (3 input channels, 4 classes, 256 x 256).  Each round runs, alternating:
  (a) examples/infer_c.c (compiled into a temporary directory, run as a subprocess, no Python in it): prepare, a batch-64
      forward with plain calls and replayed from its own CUDA graph (ms per image; logits + labels written), and the
      batch-1 latency of a graph replay (logits + labels); CUDA events, mean over --reps calls (10x that at batch 1);
  (b) UNet_UAPS.predict_graphed in this process: batch 64 (ms per image) and batch 1 (ms per call, which includes the
      copy of the input into the graph's static buffer), CUDA events over the same counts; and the Python plan build
      (fold + 23 PackedConv, what prepare replaces), host clock around a synchronised build.
Before timing, the C program's logits and labels are compared with predict's.  Medians over the rounds with the spread.
The batch-64 working set (about 0.5 GB of activations) exceeds the 126 MB L2.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_ensemble import event_ms, gpu_info, summary  # noqa: E402

CIN, C, H, W, B = 3, 4, 256, 256, 64


def build_example(tmp: str) -> str:
    from uaps_b200.build import NVCC
    libdir = os.path.join(ROOT, "uaps_b200", "lib")
    exe = os.path.join(tmp, "infer_c")
    r = subprocess.run([NVCC, "-O2", "-Wno-deprecated-gpu-targets", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "infer_c.c"), "-L", libdir, "-luaps_b200", "-Xlinker",
                        f"-rpath,{libdir}", "-o", exe], capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit(f"building examples/infer_c.c failed:\n{r.stdout}{r.stderr}")
    return exe


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_infer_c.py measures the B200: no CUDA device found")
    from uaps_b200.unet import UNet_UAPS, inference_params
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = UNet_UAPS(CIN, C).to(dev).eval()
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    x = torch.randn(B, CIN, H, W, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    x1 = x[:1].clone()

    with tempfile.TemporaryDirectory() as tmp:
        exe = build_example(tmp)
        files = {k: os.path.join(tmp, k + ".bin") for k in ("params", "x", "logits", "labels")}
        inference_params(model).cpu().numpy().tofile(files["params"])
        x.cpu().numpy().tofile(files["x"])
        cmd = [exe, files["params"], str(CIN), str(C), files["x"], str(B), str(H), str(W), files["logits"], files["labels"]]

        def run_c(bench: bool):
            r = subprocess.run(cmd + (["--bench", str(a.reps)] if bench else []), capture_output=True, text=True, timeout=600)
            if r.returncode != 0:
                raise SystemExit(f"infer_c failed:\n{r.stdout}{r.stderr}")
            return json.loads(r.stdout.strip().splitlines()[-1]) if bench else None

        run_c(False)
        want = model.predict(x)
        z = torch.from_numpy(np.fromfile(files["logits"], dtype=np.float32).reshape(B, C, H, W))
        y = torch.from_numpy(np.fromfile(files["labels"], dtype=np.uint8).reshape(B, H, W))
        parity = {"logits_bitwise_equal": bool(torch.equal(z, want.cpu())),
                  "labels_equal": bool(torch.equal(y, torch.softmax(want, 1).argmax(1).to(torch.uint8).cpu()))}

        def plan_build_ms():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model._infer_plan = None
            model._inference_plan()
            torch.cuda.synchronize()
            return (time.perf_counter() - t0) * 1e3

        for _ in range(3):                                    # capture both graphs, lazy initialisation
            model.predict_graphed(x)
            model.predict_graphed(x1)
        samples = {k: [] for k in ("c_prepare_ms", "c_b64_ms_per_image", "c_b64_graph_ms_per_image", "c_b1_graph_ms",
                                   "py_plan_build_ms", "py_b64_graph_ms_per_image", "py_b1_graph_ms")}
        for _ in range(a.rounds):
            res = run_c(True)
            samples["c_prepare_ms"].append(res["prepare_ms"])
            samples["c_b64_ms_per_image"].append(res["batch_ms_per_image"])
            samples["c_b64_graph_ms_per_image"].append(res["batch_graph_ms_per_image"])
            samples["c_b1_graph_ms"].append(res["batch1_graph_ms"])
            samples["py_plan_build_ms"].append(plan_build_ms())
            model.predict_graphed(x)                          # the plan is new: re-capture outside the timed window
            model.predict_graphed(x1)
            samples["py_b64_graph_ms_per_image"].append(event_ms(lambda: model.predict_graphed(x), a.reps) / B)
            samples["py_b1_graph_ms"].append(event_ms(lambda: model.predict_graphed(x1), 10 * a.reps))

    out = {"bench": "f7_c_infer", "gpu": gpu_info(), "shape": [B, CIN, H, W], "classes": C, "reps": a.reps,
           "rounds": a.rounds, "parity_with_predict": parity, "results": {k: summary(v) for k, v in samples.items()}}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
