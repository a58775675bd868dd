#!/usr/bin/env python
"""Ensemble uncertainty inference through the C ABI on one B200 (DESIGN.md f8): prints one JSON line and, with --out,
writes it.

    python tools/bench_uncertainty_c.py [--out profiles/f8_c_uncertainty_b200.json] [--reps 50] [--rounds 5]

Two shapes: NEU (64 x 3 x 256 x 256, 4 classes, 3 auxiliary decoders: K = 4, the reference network) and KoSDD2
(32 x 3 x 240 x 640, 2 classes, 4 auxiliary decoders: K = 5, which adds the fresh-draw perturbation launches of
decoder 4), each also at batch 1.  Each round runs, alternating:
  (a) examples/uncertainty_c.c (compiled into a temporary directory, run as a subprocess, no Python in it): prepare, a
      batch forward with plain calls and replayed from its own CUDA graph (ms per image; labels + uncertainty +
      per-image uncertainty written), and the batch-1 latency of a graph replay; CUDA events, mean over --reps calls
      (10x that at batch 1);
  (b) UNet_UAPS.predict_uncertainty_graphed in this process at the same batch (ms per image) and at batch 1 (ms per
      call, which includes drawing the host random numbers and copying them and the input into the graph's static
      buffers), CUDA events over the same counts; and the Python plan build (_inference_plan() and _aux_plan(a) for
      every decoder: fold + PackedConv, what prepare replaces), host clock around a synchronised build.
Before timing, the C program's outputs are asserted bitwise equal to predict_uncertainty(x, seed=...) from the same
draws.  Medians over the rounds with the spread.  Both batch working sets (over 1.5 GB of activations) exceed the
126 MB L2.
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

CONFIGS = [("neu", 64, 3, 256, 256, 4, 3), ("kosdd2", 32, 3, 240, 640, 2, 4)]   # name, B, cin, H, W, C, n_aux
SEED = 1234


def build_example(tmp: str) -> str:
    from uaps_b200.build import NVCC
    libdir = os.path.join(ROOT, "uaps_b200", "lib")
    exe = os.path.join(tmp, "uncertainty_c")
    r = subprocess.run([NVCC, "-O2", "-Wno-deprecated-gpu-targets", "-I", os.path.join(ROOT, "include"),
                        os.path.join(ROOT, "examples", "uncertainty_c.c"), "-L", libdir, "-luaps_b200", "-Xlinker",
                        f"-rpath,{libdir}", "-o", exe], capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit(f"building examples/uncertainty_c.c failed:\n{r.stdout}{r.stderr}")
    return exe


def bench_config(exe, tmp, name, B, cin, H, W, C, n_aux, reps, rounds):
    from uaps_b200.unet import UNet_UAPS, inference_params
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    model = UNet_UAPS(cin, C, n_aux=n_aux).to(dev).eval()
    with torch.no_grad():
        for m in model.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.normal_(0, 0.1)
                m.running_var.uniform_(0.5, 1.5)
    x = torch.randn(B, cin, H, W, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    x1 = x[:1].clone()

    files = {k: os.path.join(tmp, f"{name}_{k}.bin") for k in ("params", "x", "draws", "labels", "unc", "img")}
    inference_params(model, ensemble=True).cpu().numpy().tofile(files["params"])
    x.cpu().numpy().tofile(files["x"])
    model._ensemble_draws(SEED).tofile(files["draws"])
    cmd = [exe, files["params"], str(cin), str(C), str(n_aux), files["x"], files["draws"], str(B), str(H), str(W),
           files["labels"], files["unc"], files["img"]]

    def run_c(bench: bool):
        r = subprocess.run(cmd + (["--bench", str(reps)] if bench else []), capture_output=True, text=True, timeout=900)
        if r.returncode != 0:
            raise SystemExit(f"uncertainty_c failed:\n{r.stdout}{r.stderr}")
        return json.loads(r.stdout.strip().splitlines()[-1]) if bench else None

    run_c(False)
    want = model.predict_uncertainty(x, seed=SEED)
    got = (np.fromfile(files["labels"], dtype=np.uint8).reshape(B, H, W),
           np.fromfile(files["unc"], dtype=np.float32).reshape(B, H, W),
           np.fromfile(files["img"], dtype=np.float32).reshape(B))
    parity = {k: bool(torch.equal(torch.from_numpy(g), w.cpu()))
              for k, g, w in zip(("labels", "uncertainty", "image_uncertainty"), got, want)}
    if not all(parity.values()):
        raise SystemExit(f"{name}: the C program's outputs differ from predict_uncertainty: {parity}")

    def plan_build_ms():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model._infer_plan = None
        model._inference_plan()
        for a in range(1, n_aux + 1):
            model._aux_plan(a)
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    graphed = lambda inp: model.predict_uncertainty_graphed(inp, seed=SEED)    # noqa: E731
    for _ in range(3):                                    # capture both graphs, lazy initialisation
        graphed(x)
        graphed(x1)
    samples = {k: [] for k in ("c_prepare_ms", "c_batch_ms_per_image", "c_batch_graph_ms_per_image", "c_b1_graph_ms",
                               "py_plan_build_ms", "py_batch_graph_ms_per_image", "py_b1_graph_ms")}
    for _ in range(rounds):
        res = run_c(True)
        samples["c_prepare_ms"].append(res["prepare_ms"])
        samples["c_batch_ms_per_image"].append(res["batch_ms_per_image"])
        samples["c_batch_graph_ms_per_image"].append(res["batch_graph_ms_per_image"])
        samples["c_b1_graph_ms"].append(res["batch1_graph_ms"])
        samples["py_plan_build_ms"].append(plan_build_ms())
        graphed(x)                                        # the plan is new: re-capture outside the timed window
        graphed(x1)
        samples["py_batch_graph_ms_per_image"].append(event_ms(lambda: graphed(x), reps) / B)
        samples["py_b1_graph_ms"].append(event_ms(lambda: graphed(x1), 10 * reps))
    return {"shape": [B, cin, H, W], "classes": C, "n_aux": n_aux, "K": 1 + n_aux,
            "parity_with_predict_uncertainty": parity, "results": {k: summary(v) for k, v in samples.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_uncertainty_c.py measures the B200: no CUDA device found")
    with tempfile.TemporaryDirectory() as tmp:
        exe = build_example(tmp)
        configs = {c[0]: bench_config(exe, tmp, *c, a.reps, a.rounds) for c in CONFIGS}
    out = {"bench": "f8_c_uncertainty", "gpu": gpu_info(), "seed": SEED, "reps": a.reps, "rounds": a.rounds,
           "configs": configs}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
