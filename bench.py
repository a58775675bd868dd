#!/usr/bin/env python
"""bench.py -- the UAPS unlabeled-batch hot path on B200, one JSON line (contract: task brief (4)).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config neu|dagm|kosdd2]
                    [--no-train-step] [--no-sweep] [--no-other-configs] [--dump-outputs DIR]

--steps K sets the timed steps of the headline blocks only: the headline loss and the headline configuration's training
iteration.  The other configurations, the sweep, the inference block and the host-logits footnote keep their own fixed
counts (the footnote takes K clamped to 3..10).

--dump-outputs DIR writes, after the timed steps, what the headline loss path returned in its last step as
DIR/<name>.npy (see DUMP_SAMPLE).  Its inputs depend only on the arguments and its outputs are bitwise reproducible, so
two builds can be compared output for output.
The training iteration is not dumped: it sums its BatchNorm statistics with atomics, whose order varies, so it differs run
to run in the last bits, and the iterations amplify that.

Headline workload (BASELINE.json configs[1] at the shape of configs[2]'s unlabeled batch): the fused
pseudo-label + KL-uncertainty + weighted CE/Dice loss, forward + backward, K=4 decoders, C=4
classes, 64 x 256x256 pixels per GPU (268 MB of fp32 logits, > the 126 MB L2).  One "step" = pass 1 +
fold/finalize + pass 2 over one batch (3 launches chained by programmatic dependent launch).  metric =
pixels/s over all ranks (weak scaling: every rank has its own batch; the <=70-double partial-sum vector is
exchanged between the passes inside the fold kernel, through NVLink peer-memory mailboxes).

  value     : logits resident in HBM, C-ABI calls timed with CUDA events on the launching stream.
  roofline  : the dominant kernel (pass 2: 8*K*C algorithmic bytes / pixel) against the measured HBM
              copy bandwidth in MEASURED_PEAKS.json; per-kernel numbers under "kernels".
  e2e       : the path's real host boundary -- host IMAGES in, loss scalar out -- through the public API
              (UAPSTrainer.step: both forwards of the K-decoder U-Net, both fused losses, backward, Adam; captured
              CUDA graph), in the headline metric's unit: unlabeled pixels per second through the whole iteration.
              The H2D copy of the batch and the D2H read of the loss are inside the timed region.
              ("e2e_host_logits" keeps round 1's figure -- the loss API fed from pinned host LOGITS -- as a footnote:
              it measures PCIe, because in UAPS the logits never come from the host.)
  train_step: the co-headline (BASELINE metric "UAPS train iters/s"): iters/s, images/s, TFLOP/iteration against the
              measured sustained bf16 peak, and the CPU arm's ratio.
  configs   : the same two measurements (loss roofline + training iteration) on the DAGM- and KoSDD2-shaped
              configurations of BASELINE.json (configs[3], configs[4]: 512x512 C=2 32+32; 240x640 C=2 K=5 32+32).
  sweep     : points of configs[1]'s sweep (K 2-6, C 2-4, 200x200 .. 1024x1024, batch 8-256), each beside the reference's
              expressions as torch-eager CUDA ops on the same GPU (the incumbent GPU path).
  cpu_baseline : the oracle (restated reference expressions, torch CPU) on the box's host cores.

--impl reference times the reference's CPU implementation of the same path (the oracle port; the
reference itself is pure Python over torch and its loss section is inline code that cannot be
imported -- see DESIGN.md) on all host cores, on the same workload and step/warm-up counts.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# BASELINE.json configs[2], [3], [4]: per-GPU batch (labeled + unlabeled), image shape as it passes the 4x-pooled U-Net
CONFIGS = {
    "neu": dict(K=4, C=4, B=64, H=256, W=256, cin=3,
                what="NEU-Seg-shaped: 200x200 resized to 256x256 as the reference does (utilities/dataloaders.py:98), 4 classes, 64+64"),
    "dagm": dict(K=4, C=2, B=32, H=512, W=512, cin=1,
                 what="DAGM-shaped 512x512 grayscale, 2 classes, 32+32"),
    "kosdd2": dict(K=5, C=2, B=32, H=240, W=640, cin=3,
                   what="KolektorSDD2-shaped 232x640 padded to 240x640, 2 classes, 5 decoders (4th aux: FeatureNoise, fresh draw), 32+32"),
}
CW1 = CW2 = 0.1
CPU_TRAIN_B = 4                        # bounded CPU sample of the full iteration: 4 + 4 images
FT = (16, 32, 64, 128, 256)
DUMP_SAMPLE = 1 << 22                  # --dump-outputs keeps this many elements of a larger output (16 MB of float32)
DUMP_MAX_BYTES = 64 << 20


def dump_sample(ts):
    """The tensors `ts` flattened and concatenated as a host array, or, when that is longer than DUMP_SAMPLE, the
    DUMP_SAMPLE elements at a fixed set of positions (drawn with seed 0, in increasing order)."""
    total = sum(t.numel() for t in ts)
    if total <= DUMP_SAMPLE:
        return torch.cat([t.detach().reshape(-1) for t in ts]).cpu().numpy()
    idx = np.sort(np.random.default_rng(0).choice(total, DUMP_SAMPLE, replace=False))
    out, start = [], 0
    for t in ts:
        sel = idx[(idx >= start) & (idx < start + t.numel())] - start
        out.append(t.detach().reshape(-1)[torch.from_numpy(sel).to(t.device)].cpu())
        start += t.numel()
    return torch.cat(out).numpy()


def write_dump(path, arrays):
    """arrays: {name: float32 / float64 array} -> path/<name>.npy."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values()), {k: a.dtype for k, a in arrays.items()}
    nbytes = sum(a.nbytes for a in arrays.values())
    assert nbytes <= DUMP_MAX_BYTES, nbytes
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def workload_name(c):
    return f"fused_loss_fwd_bwd K={c['K']} C={c['C']} B={c['B']}/gpu {c['H']}x{c['W']} fp32-logits"


def line_config(c):
    """The `config` object both arms print -- literally the same dict."""
    return {"workload": workload_name(c), "K": c["K"], "C": c["C"], "H": c["H"], "W": c["W"], "batch_per_gpu": c["B"],
            "l2": "inputs (logits + gradients per GPU) larger than the 126 MB L2; no flush"}


def model_flops_per_image(cin, C, K, H, W):
    """Forward FLOPs (2 x MACs) of UNet_UAPS with K decoders on one cin x H x W image (utilities/UAPS_unet.py:89-153)."""
    f = 0
    for l in range(5):
        h, w = H >> l, W >> l
        ci = cin if l == 0 else FT[l - 1]
        f += 2 * h * w * 9 * (ci * FT[l] + FT[l] * FT[l])
    dec = 0
    for i in range(1, 5):
        c1, c2 = FT[5 - i], FT[4 - i]
        hl, wl = H >> (5 - i), W >> (5 - i)
        h, w = H >> (4 - i), W >> (4 - i)
        dec += 2 * hl * wl * c1 * c2                            # conv1x1 at the low resolution
        dec += 2 * h * w * 9 * (2 * c2 * c2 + c2 * c2)          # ConvBlock(2 c2 -> c2 -> c2)
    dec += 2 * H * W * 9 * FT[0] * C                            # out_conv
    return f + K * dec


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", 1400.0)), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, 1400.0, "fallback (B200_PROFILING.md: 6.65 TB/s, ~1.4 PFLOP/s sustained)"


def ncu_traffic():
    """DRAM bytes per pass-2 launch from the committed ncu --set full capture (profiles/), or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "loss_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s in sm if mx and s > 0.5 * mx] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- CPU / incumbent legs (the only places that touch oracle/) ------------------------------------------------
def eager_cuda_loss(dev, K, C, B, H, W, steps=3, warmup=1):
    """The reference's own loss expressions (the oracle restatement, bit-identical to the executed reference lines) as
    torch-eager ops ON THE SAME B200, fwd + bwd: the incumbent GPU number the fused kernels replace."""
    from oracle.uaps_loss_ref import unlabeled_loss_ref
    gen = torch.Generator(device=dev).manual_seed(1337)
    z = [(torch.randn(B, C, H, W, generator=gen, device=dev) * 2).requires_grad_(True) for _ in range(K)]
    mix_w = np.random.default_rng(1337).dirichlet(np.ones(K))

    def one():
        for t in z:
            t.grad = None
        unlabeled_loss_ref(z, mix_w, CW1, CW2)["loss_u"].backward()

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    del z
    torch.cuda.empty_cache()
    return ms


def cpu_loss(c, batch, steps, warmup, threads):
    """The oracle's unlabeled loss fwd+bwd on CPU torch (the reference's expressions): (pixels/s, s/step)."""
    from oracle.uaps_loss_ref import unlabeled_loss_ref
    torch.set_num_threads(threads)
    K, C, H, W = c["K"], c["C"], c["H"], c["W"]
    g = torch.Generator().manual_seed(1337)
    z = [(torch.randn(batch, C, H, W, generator=g) * 2).requires_grad_(True) for _ in range(K)]
    mix_w = np.random.default_rng(1337).dirichlet(np.ones(K))
    times = []
    for i in range(warmup + steps):
        for t in z:
            t.grad = None
        t0 = time.perf_counter()
        out = unlabeled_loss_ref(z, mix_w, CW1, CW2)
        out["loss_u"].backward()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    px = batch * H * W
    return px * len(times) / sum(times), sum(times) / len(times)


def cpu_train_step(c, steps, warmup, threads, batch=CPU_TRAIN_B):
    """The reference's full iteration on CPU: oracle functional U-Net + oracle losses + Adam; iters/s.
    The oracle network is the reference's K = 4 model, so a K = 5 configuration is timed with K = 4 on the CPU side
    (it flatters the CPU arm by one decoder; stated in the sample string)."""
    from oracle.unet_ref import feature_shapes, synthetic_rand, synthetic_state_dict, unet_uaps_ref
    from oracle.uaps_loss_ref import supervised_loss_ref, unlabeled_loss_ref
    torch.set_num_threads(threads)
    C, H, W, cin = c["C"], c["H"], c["W"], c["cin"]
    sd = synthetic_state_dict(cin, C)
    params = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    full = {**sd, **params}
    opt = torch.optim.Adam(list(params.values()), lr=1e-3)
    g = torch.Generator().manual_seed(1337)
    xl, xu = torch.randn(batch, cin, H, W, generator=g), torch.randn(batch, cin, H, W, generator=g)
    yl = torch.randint(0, C, (batch, H, W), generator=g)
    rand = synthetic_rand(feature_shapes(batch, H, W))
    mix_w = np.random.default_rng(1337).dirichlet(np.ones(4))
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ol = unet_uaps_ref(xl, full, rand)[:4]
        ou = unet_uaps_ref(xu, full, rand)[:4]
        loss = supervised_loss_ref(ol, yl)["supervised_loss"] + unlabeled_loss_ref(ou, mix_w, CW1, CW2)["loss_u"]
        opt.zero_grad()
        loss.backward()
        opt.step()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return len(times) / sum(times)


def cpu_train_block(c, threads, steps=2, warmup=1):
    its = cpu_train_step(c, steps, warmup, threads)
    return {"iters_per_s": its, "images_per_s": 2 * CPU_TRAIN_B * its, "unlabeled_pixels_per_s": CPU_TRAIN_B * c["H"] * c["W"] * its,
            "cores": threads, "kind": "port",
            "sample": f"oracle U-Net (K=4) + oracle losses + autograd + Adam on CPU torch, {CPU_TRAIN_B}+{CPU_TRAIN_B} images "
                      f"{c['cin']}x{c['H']}x{c['W']} C={c['C']}, {steps} timed iterations"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    c = CONFIGS[args.config]
    threads = os.cpu_count() or 1
    # the SAME sample as the GPU arm's step (B x H x W pixels per step) and the same step / warm-up counts
    pxs, sec = cpu_loss(c, c["B"], args.steps, args.warmup, threads)
    line = {
        "impl": "reference", "metric": "fused_pl_kl_loss_pixels_per_s", "value": pxs, "unit": "pixels/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": line_config(c),
        "cpu_baseline": {"value": pxs, "unit": "pixels/s", "cores": threads, "kind": "port",
                         "sample": f"oracle (reference expressions, torch CPU) fwd+bwd on {c['B']}x{c['H']}x{c['W']} px per step "
                                   "(the GPU arm's whole per-GPU step)"},
        "gpu_launches": 0,
    }
    e2e_px = pxs
    if not args.no_train_step:
        try:
            blk = cpu_train_block(c, threads)
            line["train_step"] = {**blk, "unit": "iters/s"}
            e2e_px = blk["unlabeled_pixels_per_s"]
            if not args.no_other_configs:
                line["configs"] = {}
                for name, oc in CONFIGS.items():
                    if name == args.config:
                        continue
                    p2, _ = cpu_loss(oc, 2, 2, 1, threads)
                    line["configs"][name] = {"loss": {"pixels_per_s": p2, "sample": f"2x{oc['H']}x{oc['W']} px per step"},
                                             "train_step": cpu_train_block(oc, threads)}
        except Exception as e:                                   # the headline line must still print
            line["train_step"] = {"error": repr(e)[:200]}
    # e2e of this arm: the same boundary as the GPU arm's e2e (host images in -> one full training iteration ->
    # loss out), in unlabeled pixels/s; everything already lives in host memory, so no copies
    line["e2e"] = {"value": e2e_px, "unit": "pixels/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "api": "reference iteration on CPU (UAPS_train.py:177-292 as restated by oracle/), unlabeled pixels/s"
                   if e2e_px != pxs else "loss only (train step disabled)"}
    print(json.dumps(line), flush=True)


# ---- GPU arm ---------------------------------------------------------------------------------------------------
def loss_bench(c, dev, lib, L, group, world, rank, xchg, steps, warmup, seed_off=0, dump=None):
    """Device-resident fused loss fwd+bwd through the C ABI: (ms_total, t_pass1, t_pass2, n_events).  `dump` (a dict)
    receives the last step's scalars, partial sums and a sample of the logits' gradient."""
    import torch.distributed as dist
    K, C, B, H, W = c["K"], c["C"], c["B"], c["H"], c["W"]
    N = B * H * W
    gen = torch.Generator(device=dev).manual_seed(1337 + rank + seed_off)
    z = [torch.randn(B, C, H, W, generator=gen, device=dev) * 2 for _ in range(K)]
    dz = [torch.empty_like(t) for t in z]
    mix_w = np.random.default_rng(1337).dirichlet(np.ones(K))
    ws = torch.zeros(lib.uaps_loss_workspace_bytes(K, C), dtype=torch.uint8, device=dev)
    sums = torch.empty(lib.uaps_loss_sums_count(K, C), dtype=torch.float64, device=dev)
    sc = torch.empty(lib.uaps_loss_scalars_count(K, C), dtype=torch.float32, device=dev)
    go = torch.zeros_like(sc)
    go[0] = 1.0
    zp, dzp, w_arr = L.ptr_array(z), L.ptr_array(dz), L.float_array(mix_w)
    st = L.stream_ptr()

    def step(ev=None):
        if world == 1:          # single rank: fold + finalize fused into one launch behind pass 1
            L.check(lib.uaps_loss_pass1_scalars(zp, K, B, C, H * W, w_arr, None, ws.data_ptr(), sums.data_ptr(), None, None, 0,
                                                CW1, CW2, sc.data_ptr(), None, st), "pass1")
        elif xchg is not None:  # fold + peer-memory exchange + finalize in one launch
            L.check(lib.uaps_loss_pass1_exchange(zp, K, B, C, H * W, w_arr, None, ws.data_ptr(), sums.data_ptr(), None, None, 0,
                                                 xchg.ptrs, rank, world, xchg.next_epoch(), N * world, CW1, CW2, sc.data_ptr(),
                                                 None, None, st), "pass1")
        else:
            L.check(lib.uaps_loss_pass1(zp, K, B, C, H * W, w_arr, None, ws.data_ptr(), sums.data_ptr(), None, None, 0, st), "pass1")
            dist.all_reduce(sums, group=group)
            L.check(lib.uaps_loss_finalize(sums.data_ptr(), K, C, N * world, CW1, CW2, 0, sc.data_ptr(), st), "finalize")
        if ev: ev[0].record()
        L.check(lib.uaps_loss_pass2(zp, K, B, C, H * W, w_arr, None, sc.data_ptr(), go.data_ptr(), dzp, 0, None, st), "pass2")
        if ev: ev[1].record()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warmup):
        step()
    # Per-kernel events on every EV_EVERY-th step only (three records: start, after pass 1 + fold/finalize, end): an event
    # record between two launches cancels their programmatic-dependent-launch overlap, so the other steps run as the
    # library is used in a training loop.  `value` is from the outer pair of events around all K steps.
    EV_EVERY = 4
    evs = {i: [torch.cuda.Event(enable_timing=True) for _ in range(3)] for i in range(0, steps, EV_EVERY)}
    barrier()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for i in range(steps):
        ev = evs.get(i)
        if ev:
            ev[0].record()
        step(ev[1:] if ev else None)
    t_end.record()
    barrier()
    ms_total = t_start.elapsed_time(t_end)
    t1 = sum(e[0].elapsed_time(e[1]) for e in evs.values()) / len(evs)      # pass 1 + fold/finalize (+ exchange)
    t2 = sum(e[1].elapsed_time(e[2]) for e in evs.values()) / len(evs)      # pass 2
    t = torch.tensor([ms_total, t1, t2], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, t1, t2 = t.tolist()
    if dump is not None:
        dump.update(loss_scalars=sc.cpu().numpy(), loss_sums=sums.cpu().numpy(), loss_grad_logits=dump_sample(dz))
    del z, dz
    return ms_total, t1, t2, len(evs), EV_EVERY


def loss_roofline(c, ms_total, t1, t2, steps, world, peak, peak_src):
    K, C, N = c["K"], c["C"], c["B"] * c["H"] * c["W"]
    ms_step = ms_total / steps
    bytes1, bytes2 = 4 * K * C * N, 8 * K * C * N
    ach1, ach2 = bytes1 / (t1 * 1e-3) / 1e9, bytes2 / (t2 * 1e-3) / 1e9
    vec = "VEC=4" if K * C <= 12 else ("VEC=2" if K * C <= 24 else "VEC=1")     # fused_loss.cu:pick_impl / dispatch
    roof = {"bound": "hbm", "kernel": f"loss_pass2_kernel<K={K},C={C},{vec},PF> (uaps_loss_pass2)", "achieved": ach2, "peak": peak,
            "unit": "GB/s", "frac": ach2 / peak, "peak_source": peak_src, "algorithmic_bytes_per_launch": bytes2,
            "fwd_bwd_frac": (bytes1 + bytes2) / (ms_step * 1e-3) / 1e9 / peak}
    kernels = {"pass1_fold_finalize" + ("_exchange" if world > 1 else ""):
                   {"ms": t1, "GBps": ach1, "frac": ach1 / peak, "algorithmic_bytes": bytes1},
               "pass2": {"ms": t2, "GBps": ach2, "frac": ach2 / peak, "algorithmic_bytes": bytes2}}
    return roof, kernels, N * world * steps / (ms_total * 1e-3), ms_step


def e2e_host_logits(c, dev, group, world, mix_w, steps):
    """Round 1's e2e, kept as a footnote: the loss API fed from pinned host LOGITS (PCIe-bound by construction)."""
    import torch.distributed as dist
    from uaps_b200.losses import uaps_unlabeled_loss
    K, C, B, H, W = c["K"], c["C"], c["B"], c["H"], c["W"]
    zh = [torch.randn(B, C, H, W).mul_(2).pin_memory() for _ in range(K)]
    zd = [torch.empty((B, C, H, W), device=dev).requires_grad_(True) for _ in range(K)]
    out_host = torch.empty(3, dtype=torch.float32).pin_memory()

    def one():
        for hsrc, d in zip(zh, zd):
            d.grad = None
            d.data.copy_(hsrc, non_blocking=True)
        loss, ps, unc, _, _ = uaps_unlabeled_loss(zd, mix_w, CW1, CW2, group=group)
        loss.backward()
        out_host.copy_(torch.stack([loss.detach(), ps.detach(), unc.detach()]), non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(2):
        one()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item()
    return {"value": B * H * W * world * steps / (ms * 1e-3), "unit": "pixels/s", "h2d_bytes_per_step": 4 * K * C * B * H * W,
            "d2h_bytes_per_step": 12, "steps": steps, "api": "uaps_b200.losses.uaps_unlabeled_loss + backward, pinned host logits"}


def sharded_equals_full(dev, group, world, rank):
    """N > 1 correctness, outside any timed region: every rank evaluates the loss on ITS shard through the multi-rank
    path (sums exchanged between the passes) and on the all-gathered FULL batch through the single-rank path; the
    scalars must agree to 1e-6, the pseudo-labels exactly, and the shard's gradient with its slice of the full one."""
    import torch.distributed as dist
    from uaps_b200.losses import uaps_unlabeled_loss
    K, C, B, H, W = 4, 4, 4, 128, 128
    gen = torch.Generator(device=dev).manual_seed(4242 + rank)
    mix_w = np.random.default_rng(7).dirichlet(np.ones(K))
    z = [(torch.randn(B, C, H, W, generator=gen, device=dev) * 2).requires_grad_(True) for _ in range(K)]
    loss, ps, unc, pseudo, _ = uaps_unlabeled_loss(z, mix_w, CW1, CW2, group=group, return_pseudo=True)
    loss.backward()
    full = []
    for t in z:
        parts = [torch.empty_like(t.detach()) for _ in range(world)]
        dist.all_gather(parts, t.detach().contiguous(), group=group)
        full.append(torch.cat(parts, 0).requires_grad_(True))
    lf, pf, uf, pseudo_f, _ = uaps_unlabeled_loss(full, mix_w, CW1, CW2, group=None, return_pseudo=True)
    lf.backward()
    rel = lambda a, b: abs(float(a.detach()) - float(b.detach())) / max(abs(float(b.detach())), 1e-30)
    errs = [rel(loss, lf), rel(ps, pf), rel(unc, uf)]
    sl = slice(rank * B, (rank + 1) * B)
    gerr = max(float((a.grad - b.grad[sl]).abs().max() / b.grad[sl].abs().max()) for a, b in zip(z, full))
    ok = max(errs) <= 1e-6 and gerr <= 1e-5 and bool(torch.equal(pseudo, pseudo_f[sl]))
    flag = torch.tensor([1.0 if ok else 0.0, max(errs), gerr], dtype=torch.float64, device=dev)
    mn = flag.clone()
    dist.all_reduce(mn, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
    return {"ok": bool(mn[0].item() == 1.0), "max_scalar_rel_err": flag[1].item(), "max_grad_rel_err": flag[2].item(),
            "pseudo_labels_exact": ok, "shape": f"K={K} C={C} {B}x{H}x{W} per rank, {world} ranks"}


def train_step_bench(c, dev, group, world, rank, steps: int = 8, warmup: int = 4, compute: str = "bf16", batch=None):
    """Full UAPS iteration (UAPS_train.py:159-314 body): host batch in, loss scalar out, inside the timed region."""
    import torch.distributed as dist
    from uaps_b200.train import UAPSConfig, UAPSTrainer
    from uaps_b200.unet import UNet_UAPS
    K, C, H, W, cin = c["K"], c["C"], c["H"], c["W"], c["cin"]
    batch = batch or c["B"]
    torch.manual_seed(1337)
    model = UNet_UAPS(cin, C, n_aux=K - 1, compute=compute).to(dev)
    trainer = UAPSTrainer(model, UAPSConfig(num_classes=C), group=group)
    gen = torch.Generator().manual_seed(1337 + rank)
    xl_h = torch.randn(batch, cin, H, W, generator=gen).pin_memory()
    xu_h = torch.randn(batch, cin, H, W, generator=gen).pin_memory()
    yl_h = torch.randint(0, C, (batch, H, W), generator=gen).pin_memory()
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()

    def it():
        # pinned host batch in (H2D on the trainer's copy stream, overlapping the previous iteration's kernels),
        # loss scalar out (D2H) -- both inside the timed region, every step
        out = trainer.step_host(xl_h, yl_h, xu_h)
        loss_h.copy_(out["loss"], non_blocking=True)

    for _ in range(warmup):
        it()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        it()
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / steps
    _, tf_peak, peak_src = measured_peaks()
    flop = 3.0 * model_flops_per_image(cin, C, K, H, W) * 2 * batch            # fprop + dgrad + wgrad, labeled + unlabeled
    tfs = flop / (ms * 1e-3) / 1e12
    mode = ("captured CUDA graph" if trainer._graphs else "device-state eager") if trainer.state is not None else "host scalars, eager launches"
    out = {"iters_per_s": 1e3 / ms, "ms_per_iter": ms, "steps": steps, "images_per_s": 2 * batch * world * 1e3 / ms,
           "unlabeled_pixels_per_s": batch * H * W * world * 1e3 / ms, "unit": "iters/s", "loss": float(loss_h),
           "h2d_bytes_per_iter": xl_h.numel() * 4 * 2 + yl_h.numel() * 8, "d2h_bytes_per_iter": 4,
           "tflop_per_iter_per_gpu": flop / 1e12,
           "roofline": {"bound": "tensor", "achieved": tfs, "peak": tf_peak, "unit": "TFLOP/s", "frac": tfs / tf_peak,
                        "peak_source": peak_src + " bf16_tflops_sustained",
                        "note": "whole iteration against the dense-GEMM peak; 60 % of the FLOPs sit in 16/32-channel layers that are "
                                "HBM-bound by construction (arithmetic intensity 36-72 FLOP/B), see DESIGN.md"},
           "mode": mode, "skipped_updates": trainer.skipped_steps(),
           "config": f"UNet_UAPS {cin}x{H}x{W} C={C} K={K}, {batch}+{batch} images/GPU, dp{world}, host images in the timed region",
           "kernels": "bf16 channels-last: tcgen05 implicit-GEMM fprop/dgrad/wgrad, fused BN+LeakyReLU+dropout, pool/upsample, Philox "
                      "perturbations, fused losses, flat Adam (all hand-written sm_100a)" if compute == "bf16" else
                      "cuDNN fp32 (reference-precision path)"}
    del trainer, model
    torch.cuda.empty_cache()
    return out


def loss_sweep(dev, lib, L, with_eager=True, iters: int = 10):
    """Points of BASELINE configs[1]'s sweep (K 2-6, C 2-4, 200x200 .. 1024x1024, batch 8-256), device-resident, same timing
    method as the headline; beside each, the reference expressions as torch-eager CUDA ops (the incumbent)."""
    peak, _, _ = measured_peaks()
    pts = [(2, 2, 8, 200, 200), (4, 4, 8, 200, 200), (3, 3, 16, 256, 256), (4, 4, 64, 512, 512), (4, 2, 32, 512, 512),
           (5, 2, 32, 232, 640), (6, 4, 32, 512, 512), (2, 4, 128, 512, 512), (3, 2, 256, 512, 512), (2, 2, 128, 1024, 1024),
           (3, 4, 32, 1024, 1024), (4, 4, 256, 256, 256)]
    out = []
    for (k, c, b, h, w) in pts:
        z = [torch.randn(b, c, h, w, device=dev) * 2 for _ in range(k)]
        dz = [torch.empty_like(t) for t in z]
        ws = torch.zeros(lib.uaps_loss_workspace_bytes(k, c), dtype=torch.uint8, device=dev)
        sums = torch.empty(lib.uaps_loss_sums_count(k, c), dtype=torch.float64, device=dev)
        sc = torch.empty(lib.uaps_loss_scalars_count(k, c), dtype=torch.float32, device=dev)
        go = torch.zeros_like(sc); go[0] = 1.0
        zp, dzp, wa, st = L.ptr_array(z), L.ptr_array(dz), L.float_array([1.0 / k] * k), L.stream_ptr()
        n = b * h * w

        def step():
            L.check(lib.uaps_loss_pass1_scalars(zp, k, b, c, h * w, wa, None, ws.data_ptr(), sums.data_ptr(), None, None, 0,
                                                CW1, CW2, sc.data_ptr(), None, st), "p1")
            L.check(lib.uaps_loss_pass2(zp, k, b, c, h * w, wa, None, sc.data_ptr(), go.data_ptr(), dzp, 0, None, st), "p2")
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            step()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        row = {"K": k, "C": c, "B": b, "H": h, "W": w, "ms_per_step": ms, "pixels_per_s": n / (ms * 1e-3),
               "fwd_bwd_frac_of_hbm_peak": 12 * k * c * n / (ms * 1e-3) / 1e9 / peak,
               "l2": "resident" if 8 * k * c * n < 126e6 else "exceeds L2"}
        del z, dz
        if with_eager:
            # the eager path keeps ~60 intermediates of the logits' size alive for autograd: bound its batch by memory and
            # scale per pixel (it is launch- and bandwidth-bound the same way at every batch size above a few Mpx)
            be = b
            while be > 1 and 4 * k * c * be * h * w * 70 > 60e9:
                be //= 2
            try:
                ems = eager_cuda_loss(dev, k, c, be, h, w)
                epx = be * h * w / (ems * 1e-3)
                row["eager_cuda"] = {"pixels_per_s": epx, "ms_per_step": ems, "batch": be, "speedup": row["pixels_per_s"] / epx}
            except Exception as e:                       # noqa: BLE001 -- a baseline leg must not sink the bench line
                row["eager_cuda"] = {"error": repr(e)[:120]}
        out.append(row)
    return out


def inference_bench(c, dev, batch: int = 64, steps: int = 10, warmup: int = 3):
    """Row f3: validation / inference forward (UAPS_train.py:367-393) -- main decoder only, BatchNorm folded into the conv
    weights, LeakyReLU in the conv epilogue.  The reference's README quotes 4.48 ms / 256x256 image for the main decoder
    (fig_data/decoder-effect.jpg, hardware not stated); reported beside, not as vs_baseline (different metric)."""
    from uaps_b200.unet import UNet_UAPS
    C, H, W = c["C"], c["H"], c["W"]
    torch.manual_seed(1337)
    model = UNet_UAPS(3, C, compute="bf16").to(dev).eval()
    x_h = torch.randn(batch, 3, H, W).pin_memory()
    lab_h = torch.empty((batch, H, W), dtype=torch.uint8).pin_memory()

    def it():
        logits = model.predict(x_h.to(dev, non_blocking=True))
        lab_h.copy_(logits.argmax(1).to(torch.uint8), non_blocking=True)      # the label map goes back to the host

    for _ in range(warmup):
        it()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        it()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps

    # latency mode: one image per call, host image in, label map out; plain launches vs the captured CUDA graph
    x1_h = torch.randn(1, 3, H, W).pin_memory()
    lab1_h = torch.empty((1, H, W), dtype=torch.uint8).pin_memory()
    lat = {}
    for name, fn in (("launches", model.predict), ("cuda_graph", model.predict_graphed)):
        def one():
            lab1_h.copy_(fn(x1_h.to(dev, non_blocking=True)).argmax(1).to(torch.uint8), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        for _ in range(5):
            one()
        t0 = time.perf_counter()
        for _ in range(50):
            one()
        lat[name] = (time.perf_counter() - t0) / 50 * 1e3
    return {"ms_per_image": ms / batch, "images_per_s": batch * 1e3 / ms, "batch": batch, "ms_per_batch": ms,
            "latency_ms_batch1": lat,
            "config": f"UNet_UAPS.predict 3x{H}x{W} C={C}, bf16 path, eval mode, host images in / uint8 label map out",
            "published_ms_per_image": 4.48, "published_source": "reference README Fig. 9 (hardware not stated)"}


def run_ours(args):
    import torch.distributed as dist
    from uaps_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: uaps_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        group = dist.group.WORLD

    lib = L.lib()
    c = CONFIGS[args.config]
    K = c["K"]
    mix_w = np.random.default_rng(1337).dirichlet(np.ones(K))
    warmup = max(args.warmup, 3)
    peak, tf_peak, peak_src = measured_peaks()

    xchg = None
    if world > 1:                # the loss sums travel through NVLink peer mailboxes (NCCL only if that is unavailable)
        from uaps_b200.comm import exchange_for
        xchg = exchange_for(group, dev)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dump = {} if args.dump_outputs and rank == 0 else None
    # ---- headline: device-resident fused loss ------------------------------------------------------------------
    ms_total, t1, t2, n_ev, ev_every = loss_bench(c, dev, lib, L, group, world, rank, xchg, args.steps, warmup, dump=dump)
    if dump is not None:
        write_dump(args.dump_outputs, dump)
    roof, kernels, value, ms_step = loss_roofline(c, ms_total, t1, t2, args.steps, world, peak, peak_src)
    footnote = e2e_host_logits(c, dev, group, world, mix_w, max(3, min(args.steps, 10)))

    check = None
    if world > 1:
        try:
            check = sharded_equals_full(dev, group, world, rank)
        except Exception as e:                                  # noqa: BLE001
            check = {"ok": False, "error": repr(e)[:300]}

    # ---- co-headline: the training iteration (also this arm's e2e) -------------------------------------------------
    train, others = None, {}
    if not args.no_train_step:
        try:
            train = train_step_bench(c, dev, group, world, rank, steps=args.steps)
        except Exception as e:                                  # noqa: BLE001
            train = {"error": repr(e)[:300]}
        if not args.no_other_configs:
            for name, oc in CONFIGS.items():
                if name == args.config:
                    continue
                blk = {"what": oc["what"]}
                try:
                    mt, a1, a2, _, _ = loss_bench(oc, dev, lib, L, group, world, rank, xchg, 10, 3, seed_off=100)
                    r2, k2, v2, s2 = loss_roofline(oc, mt, a1, a2, 10, world, peak, peak_src)
                    blk["loss"] = {"workload": workload_name(oc), "pixels_per_s": v2, "ms_per_step": s2, "roofline": r2, "kernels": k2}
                    torch.cuda.empty_cache()
                    blk["train_step"] = train_step_bench(oc, dev, group, world, rank)
                except Exception as e:                          # noqa: BLE001
                    blk["error"] = repr(e)[:300]
                others[name] = blk
    clocks = sampler.stop() if rank == 0 else None

    sweep = None
    if world == 1 and not args.no_sweep:
        try:
            sweep = loss_sweep(dev, lib, L)
        except Exception as e:                                  # noqa: BLE001
            sweep = {"error": repr(e)[:300]}

    if rank == 0:
        traffic = ncu_traffic()
        roof["traffic"] = None if not traffic else traffic.get("pass2_dram_bytes_per_launch")
        roof["traffic_source"] = None if not traffic else traffic.get("source")
        line = {
            "metric": "fused_pl_kl_loss_pixels_per_s", "value": value, "unit": "pixels/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": line_config(c),
            "parallelism": f"dp{world}" if world > 1 else "single",
            "exchange": None if world == 1 else ("nvlink peer-memory mailboxes, fused into the fold kernel"
                                                 if xchg is not None else "nccl all-reduce of the sums"),
            "roofline": roof, "kernels": kernels,
            "kernel_events": f"sampled on every {ev_every}th step ({n_ev} of {args.steps})",
            "gpu_launches": (3 if (world == 1 or xchg is not None) else 4) * args.steps,   # pass1, fold(+exchange)+finalize, pass2
            "clocks": clocks,
            "e2e_host_logits": footnote,
        }
        if train is not None and "error" not in train:
            line["e2e"] = {"value": train["unlabeled_pixels_per_s"], "unit": "pixels/s",
                           "h2d_bytes_per_step": train["h2d_bytes_per_iter"], "d2h_bytes_per_step": train["d2h_bytes_per_iter"],
                           "api": "uaps_b200.train.UAPSTrainer.step (pinned host images + labels in, loss scalar out): the whole "
                                  "training iteration around the fused loss, unlabeled pixels/s",
                           "ms_per_step": train["ms_per_iter"]}
        else:                      # --no-train-step: the loss API from host logits is the only end-to-end number there is
            line["e2e"] = {k: footnote[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "api")}
        if check is not None:
            line["sharded_equals_full"] = check["ok"]
            line["sharded_check"] = check
        if world == 1:
            threads = os.cpu_count() or 1
            pxs, sec = cpu_loss(c, 8, 5, 1, threads)
            line["cpu_baseline"] = {"value": pxs, "unit": "pixels/s", "cores": threads, "kind": "port",
                                    "sample": f"oracle (reference expressions, torch CPU) fwd+bwd, 5 steps of 8x{c['H']}x{c['W']} px"}
            try:
                ems = eager_cuda_loss(dev, c["K"], c["C"], c["B"], c["H"], c["W"], steps=5, warmup=2)
                line["eager_cuda_baseline"] = {"value": c["B"] * c["H"] * c["W"] / (ems * 1e-3), "unit": "pixels/s", "ms_per_step": ems,
                                               "what": "reference expressions (UAPS_train.py:186-189, 223-282) as torch-eager CUDA ops on this GPU, fwd+bwd, same workload"}
            except Exception as e:                       # noqa: BLE001 -- a baseline leg must not sink the bench line
                line["eager_cuda_baseline"] = {"error": repr(e)[:200]}
            if train is not None and "error" not in train:
                try:
                    cpu = cpu_train_block(c, threads)
                    train["cpu_baseline"] = cpu
                    train["vs_cpu_images_per_s"] = train["images_per_s"] / cpu["images_per_s"]
                    for name, blk in others.items():
                        if "train_step" in blk and "error" not in blk["train_step"]:
                            ocpu = cpu_train_block(CONFIGS[name], threads)
                            blk["train_step"]["cpu_baseline"] = ocpu
                            blk["train_step"]["vs_cpu_images_per_s"] = blk["train_step"]["images_per_s"] / ocpu["images_per_s"]
                except Exception as e:                   # noqa: BLE001
                    train["cpu_baseline"] = {"error": repr(e)[:200]}
        if sweep is not None:
            line["sweep"] = sweep
        if train is not None:
            line["train_step"] = train
        if others:
            line["configs"] = others
        if world == 1 and not args.no_train_step:
            try:
                line["inference"] = inference_bench(CONFIGS["neu"], dev)
            except Exception as e:                       # noqa: BLE001
                line["inference"] = {"error": repr(e)[:200]}
        print(json.dumps(line), flush=True)
    if world > 1:
        from uaps_b200 import comm
        dist.barrier()
        comm.close_all()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline blocks (the loss and the training iteration "
                                                          "of --config); the other blocks keep fixed counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="neu", choices=sorted(CONFIGS))
    ap.add_argument("--no-train-step", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the headline loss path's outputs of its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's GPU path; --impl reference has none")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
