"""One UAPS training iteration (the loop body of UAPS_train.py:159-314) as a callable, data-parallel
over one process per GPU.

``UAPSTrainer.step(x_l, y_l, x_u)`` does what the reference does per iteration -- labeled forward
(:177), unlabeled forward (:185), supervised CE+Dice over the K decoders (:194-218), the fused
pseudo-label / KL-uncertainty / weighted CE+Dice loss (:223-277), the sigmoid ramp (:279-280), the
total (:282), ``zero_grad / backward / Adam.step`` (:285-292) -- and returns the logged scalars as
device tensors (the reference's nine ``.item()`` host syncs per iteration, :295-306, are left to
the caller, once per epoch).  With ``UAPSConfig.train_log_rows > 0`` every iteration also appends those scalars and the
labeled batch's confusion counts to a device-side training log, read once per epoch with ``log_result()``.

Three ways to run the same iteration:

* **captured** (default on the bf16 path): every per-iteration scalar the reference draws on the host -- the
  Dirichlet mix weights (:251), FeatureDropout's u (UAPS_unet.py:165), the ramp weights (:279-280), the Philox keys,
  the exchange epoch, Adam's step count -- lives in a device struct advanced by one tiny kernel
  (``uaps_step_begin``), so the ~1150 launches of an iteration are a static sequence: it is captured once per input
  shape into a CUDA graph and replayed with one ``cudaGraphLaunch``.  The first ``graph_warmup`` iterations of a
  shape run the same kernels eagerly.
* **device-state, eager** (``cfg.cuda_graph=False``): the same kernels and device-side scalars, launched one by one.
* **host** (whenever a draw is injected -- ``mix_w=``, ``rand_l=``, ``rand_u=`` -- or on the fp32 reference path):
  scalars drawn on the host and passed by value, as the reference does; this is the mode the parity tests use.

Multi-GPU (replaces ``nn.DataParallel``, UAPS_model.py:13): each rank holds B/G labeled + B/G
unlabeled images and a full parameter replica (rank 0's initial parameters and BatchNorm buffers are
broadcast at construction, as DataParallel re-broadcasts them every forward).  The loss partial sums are exchanged
inside the loss kernels so CE/Dice/mean(exp(-KL)) are taken over the WHOLE batch like the reference's
gather-to-GPU-0 does; per-pixel gradients are therefore already gradients of the global loss and
parameter gradients are SUM-all-reduced.  BatchNorm statistics stay per rank, which is what DataParallel's
per-replica BN does; dropout masks and feature noise are drawn per rank, mix weights are shared.
"""
from __future__ import annotations

import warnings
from dataclasses import dataclass
from typing import Dict, Optional

import numpy as np
import torch
import torch.distributed as dist

from . import _lib as L
from . import perturb as P
from .conv import WeightPacker, pack_scope
from .stepctx import DeviceStepState, StepContext
from .losses import uaps_supervised_loss, uaps_unlabeled_loss
from .ramps import get_current_consistency_weight
from .validate import append_row, finalize

# the scalars of the training log, in the order of its columns (then loss_ce_k[0..K-1]): the names ``step`` returns
LOG_SCALARS = ("loss", "supervised_loss", "total_loss_ce", "total_loss_dice", "ps_loss", "l_uncert")
_LOG_ERRORS = {"ranks": "the ranks logged different numbers of training iterations",
               "overflow": "more training iterations than UAPSConfig.train_log_rows since log_begin()",
               "empty": "no training iteration logged since log_begin()"}


@dataclass
class UAPSConfig:
    """The reference's argparse / module constants (UAPS_train.py:36-60, 66, 78)."""
    num_classes: int = 4
    base_lr: float = 1e-3
    consistency1: float = 0.1
    consistency2: float = 0.1
    consistency_rampup: float = 200.0
    iters_per_ramp_epoch: int = 80       # ``iter_num // 80`` (:279-280); 60/40/50 in the dataset variants
    seed: int = 1337
    optimizer: str = "uaps"              # "uaps": FlatAdam (one kernel over flat buffers); "torch": torch.optim.Adam(fused=True)
    device_state: bool = True            # per-iteration scalars on the device (bf16 path only); False: host-drawn, by value
    cuda_graph: bool = True              # capture the device-state iteration into a CUDA graph (per input shape)
    graph_warmup: int = 2                # eager iterations of a shape before it is captured
    train_log_rows: int = 0              # > 0: per-iteration training log on the device, this many iterations per epoch
                                         # (UAPSTrainer.log_begin / log_result); 0: no log, no extra launches


class FlatGradBuffer:
    """All parameter gradients as views of one contiguous fp32 buffer: zeroed with one memset,
    all-reduced with one NCCL call (14.9 MB for the 3.71 M parameters of UNet_UAPS).  Every parameter's slot starts
    on a 256-byte boundary (the kernels take 16-byte vector loads of biases and BN parameters)."""

    ALIGN = 64                            # elements: every parameter starts on a 256-byte boundary, like a torch allocation

    @classmethod
    def layout(cls, params):
        """(trainable parameters, their element offsets, total padded element count) of the flat layout."""
        params = [p for p in params if p.requires_grad]
        offsets, n = [], 0
        for p in params:
            offsets.append(n)
            n += (p.numel() + cls.ALIGN - 1) // cls.ALIGN * cls.ALIGN
        return params, offsets, n

    def __init__(self, params, flat: Optional[torch.Tensor] = None):
        """flat: an existing zero-filled fp32 buffer of the layout's size to use instead of a fresh one -- at N > 1 the
        peer-mapped allocation of ``comm.PeerGradReducer``, so the backward kernels write where the peers can read."""
        self.params, self.offsets, n = self.layout(params)
        if flat is None:
            flat = torch.zeros(n, dtype=torch.float32, device=self.params[0].device)
        elif flat.numel() != n or flat.dtype != torch.float32:
            raise RuntimeError("flat gradient buffer has the wrong size / dtype")
        self.flat = flat
        for p, off in zip(self.params, self.offsets):
            p.grad = self.flat[off:off + p.numel()].view_as(p)

    def zero(self):
        self.flat.zero_()

    def all_reduce_sum(self, group=None):
        if dist.is_initialized() and dist.get_world_size(group) > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)


class FlatAdam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr) (UAPS_train.py:112) as ONE kernel over flat buffers (uaps_adam_step).

    The parameters are re-homed into one contiguous fp32 buffer (each ``p.data`` becomes a view of it, like the
    ``.grad`` views of ``FlatGradBuffer``), so the update of all 3.71 M parameters is a single streaming launch.
    A real ``torch.optim.Optimizer`` (one param group), so ``ReduceLROnPlateau(optimizer_1, ...)`` (:113) and the
    other schedulers accept it; ``state_dict()`` / ``load_state_dict()`` speak torch.optim.Adam's format
    (state[i] = step / exp_avg / exp_avg_sq), so the reference's checkpoints (:443-450) round-trip through either optimizer.

    ``attach_state``: the step count / bias corrections (and the learning rate) then live in a ``DeviceStepState`` and the
    kernel reads them from device memory (CUDA-graph capturable iteration)."""

    def __init__(self, grads: "FlatGradBuffer", lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8):
        dev = grads.flat.device
        assert dev.type == "cuda", "uaps_b200 has no CPU path"
        defaults = dict(lr=float(lr), betas=(float(betas[0]), float(betas[1])), eps=float(eps), weight_decay=0, amsgrad=False,
                        maximize=False, foreach=None, capturable=False, differentiable=False, fused=None)
        super().__init__(list(grads.params), defaults)
        self.grads, self.params = grads, grads.params
        self.betas, self.eps = defaults["betas"], defaults["eps"]
        self._step_count_host = 0
        self._dev_state: Optional[DeviceStepState] = None
        self._lr_on_device = None
        self.flat_p = torch.zeros_like(grads.flat)     # same layout as the gradients (256-byte aligned slots, zero padding)
        with torch.no_grad():
            for p, off in zip(self.params, grads.offsets):
                view = self.flat_p[off:off + p.numel()].view_as(p)
                view.copy_(p.data)
                p.data = view                          # parameter storage now lives in the flat buffer
        self.exp_avg = torch.zeros_like(self.flat_p)
        self.exp_avg_sq = torch.zeros_like(self.flat_p)

    # ---- step count: host integer, or the device state's adam_step once attached ----------------------------------
    @property
    def step_count(self) -> int:
        if self._dev_state is not None:
            return int(self._dev_state.read().adam_step)
        return self._step_count_host

    @step_count.setter
    def step_count(self, v: int) -> None:
        self._step_count_host = int(v)
        if self._dev_state is not None:
            self._dev_state.set("adam_step", int(v))

    @property
    def lr(self) -> float:
        return float(self.param_groups[0]["lr"])

    def attach_state(self, state: DeviceStepState) -> None:
        state.set("adam_step", self._step_count_host)
        self._dev_state = state
        self.sync_lr()

    def sync_lr(self) -> None:
        """Push the param group's learning rate to the device state when a scheduler has changed it (:113)."""
        if self._dev_state is not None and self.lr != self._lr_on_device:
            self._dev_state.set("lr", self.lr)
            self._lr_on_device = self.lr

    @torch.no_grad()
    def step(self, closure=None, guard: Optional[torch.Tensor] = None, use_device_state: bool = False, reducer=None):
        """One Adam update.  use_device_state: bias corrections / lr from the attached device state (the caller has run
        ``uaps_step_begin`` this iteration); ``guard`` (a device scalar, the loss) then skips the update when it is not
        finite.  Otherwise the host step count is used, as torch.optim.Adam does.
        reducer (``comm.PeerGradReducer``, N > 1): the SAME launch first sums every rank's gradients over NVLink peer
        memory (uaps_grad_reduce_adam) -- the gradients must then NOT have been all-reduced already."""
        from . import _lib as L
        if closure is not None:
            raise RuntimeError("FlatAdam.step does not take a closure")
        st = self._dev_state if use_device_state else None
        if st is None:
            self.step_count = self.step_count + 1
            step, gptr = self._step_count_host, None
        else:
            step, gptr = 1, (None if guard is None else guard.data_ptr())
        g = self.param_groups[0]
        with L.on_device(self.flat_p.device):
            if reducer is not None:
                L.check(L.lib().uaps_grad_reduce_adam(self.flat_p.data_ptr(), reducer.grads.ptrs, self.exp_avg.data_ptr(),
                                                      self.exp_avg_sq.data_ptr(), self.flat_p.numel(), reducer.flags.ptrs,
                                                      reducer.rank, reducer.world, step, float(g["lr"]), self.betas[0],
                                                      self.betas[1], self.eps, 1.0, None if st is None else st.base, gptr,
                                                      L.stream_ptr()), "uaps_grad_reduce_adam")
                return
            L.check(L.lib().uaps_adam_step(self.flat_p.data_ptr(), self.grads.flat.data_ptr(), self.exp_avg.data_ptr(),
                                           self.exp_avg_sq.data_ptr(), self.flat_p.numel(), step, float(g["lr"]),
                                           self.betas[0], self.betas[1], self.eps, 1.0,
                                           None if st is None else st.base, gptr, L.stream_ptr()), "uaps_adam_step")

    def zero_grad(self, set_to_none: bool = False):
        self.grads.zero()

    def state_dict(self):
        state, steps = {}, self.step_count
        for i, (p, off) in enumerate(zip(self.params, self.grads.offsets)):
            n = p.numel()
            if steps > 0:
                state[i] = {"step": torch.tensor(float(steps)),
                            "exp_avg": self.exp_avg[off:off + n].view_as(p).clone(),
                            "exp_avg_sq": self.exp_avg_sq[off:off + n].view_as(p).clone()}
        group = {k: v for k, v in self.param_groups[0].items() if k != "params"}
        group["params"] = list(range(len(self.params)))
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, sd):
        steps = set()
        for i, (p, off) in enumerate(zip(self.params, self.grads.offsets)):
            n = p.numel()
            st = sd["state"].get(i)
            if st is not None:
                self.exp_avg[off:off + n].view_as(p).copy_(st["exp_avg"])
                self.exp_avg_sq[off:off + n].view_as(p).copy_(st["exp_avg_sq"])
                steps.add(int(float(st["step"])))
        if len(steps) > 1:
            # torch allows per-parameter step counts (parameters added / frozen mid-training); one kernel over a flat buffer
            # has one bias correction, so the newest count is used for all of them
            warnings.warn(f"FlatAdam: checkpoint holds per-parameter step counts {sorted(steps)}; using the largest for all")
        self.step_count = max(steps) if steps else 0
        g = sd["param_groups"][0]
        self.param_groups[0].update({k: g[k] for k in ("lr", "betas", "eps") if k in g})
        self.betas, self.eps = tuple(float(b) for b in self.param_groups[0]["betas"]), float(self.param_groups[0]["eps"])
        self.sync_lr()


def _mix64(*vals: int) -> int:
    """Deterministic 64-bit hash of a few integers (seed derivation; splitmix64 finaliser)."""
    x = 0x9E3779B97F4A7C15
    for v in vals:
        x = (x ^ (int(v) & (2 ** 64 - 1))) * 0xBF58476D1CE4E5B9 & (2 ** 64 - 1)
        x ^= x >> 31
    return x & (2 ** 64 - 1)


class _Captured:
    __slots__ = ("graph", "x_l", "y_l", "x_u", "out")


class UAPSTrainer:
    def __init__(self, model: torch.nn.Module, cfg: Optional[UAPSConfig] = None, group=None):
        if group is None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            group = dist.group.WORLD             # one process per GPU: the loss sums and the gradients span all ranks
        self.model, self.cfg, self.group = model, cfg or UAPSConfig(), group
        self.world = dist.get_world_size(group) if (group is not None and dist.is_initialized()) else 1
        self.rank = dist.get_rank(group) if self.world > 1 else 0
        # N > 1: the flat gradient buffer lives in peer-mapped memory and ONE kernel sums all ranks' gradients over NVLink
        # and applies Adam (comm.PeerGradReducer / uaps_grad_reduce_adam); NCCL's all-reduce is only the fallback
        self.reducer = None
        params, _, numel = FlatGradBuffer.layout(model.parameters())
        if self.world > 1 and self.cfg.optimizer != "torch" and params[0].is_cuda:
            from .comm import new_grad_reducer
            self.reducer = new_grad_reducer(group, params[0].device, numel)       # collective
        self.grads = FlatGradBuffer(model.parameters(), flat=None if self.reducer is None else self.reducer.grad_tensor())
        if self.cfg.optimizer == "torch":
            self.optimizer = torch.optim.Adam(self.grads.params, lr=self.cfg.base_lr, fused=True)   # :112 (library kernel)
        else:
            self.optimizer = FlatAdam(self.grads, lr=self.cfg.base_lr)                              # :112, one own kernel
        dev = self.grads.flat.device
        if self.world > 1:
            # Replicas must START identical: the gradient all-reduce only keeps identical replicas identical.  The reference's
            # DataParallel re-broadcasts GPU 0's parameters and buffers on every forward (UAPS_model.py:13); one broadcast at
            # construction is the one-process-per-GPU equivalent.
            with torch.no_grad():
                if isinstance(self.optimizer, FlatAdam):
                    dist.broadcast(self.optimizer.flat_p, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
                else:
                    for p in self.grads.params:
                        dist.broadcast(p.data, src=0, group=group)
                for b in model.buffers():
                    dist.broadcast(b, src=0, group=group)
            # per-rank host stream for the host-mode dropout / noise seeds (the replicas of the reference draw independently)
            P.manual_seed(self.cfg.seed, self.rank)
        self._iter = 0
        # identical Dirichlet draws on every rank (the reference draws once per iteration on the host, :251)
        self.rng = np.random.default_rng(self.cfg.seed)
        self.k = len(model.decoders()) if hasattr(model, "decoders") else 4
        # ---- device-resident iteration state (bf16 path, own optimizer) ----------------------------------------
        self.state: Optional[DeviceStepState] = None
        self.xchg = None
        self._graphs: Dict[tuple, _Captured] = {}
        self._warm: Dict[tuple, int] = {}
        self.packer = WeightPacker()                          # one launch re-packs every conv layer's weights per iteration
        want_dev = (self.cfg.device_state and dev.type == "cuda" and getattr(model, "compute", None) == "bf16"
                    and isinstance(self.optimizer, FlatAdam))
        if want_dev and self.world > 1:
            from .comm import new_exchange
            self.xchg = new_exchange(group, dev)              # collective; None -> no peer memory -> host mode
            want_dev = self.xchg is not None
        if want_dev:
            self.state = DeviceStepState(dev, self.cfg.base_lr)
            self.optimizer.attach_state(self.state)
            self.seed_rank = _mix64(self.cfg.seed, 0x52414E4B, self.rank)
            self.seed_shared = _mix64(self.cfg.seed, 0x53484152)
        # ---- training log (DESIGN.md f9): one row per iteration, written inside the (captured) iteration -------------
        rows = int(self.cfg.train_log_rows)
        if rows < 0:
            raise ValueError("train_log_rows must be >= 0")
        self._log_ws: Dict[tuple, torch.Tensor] = {}
        self.log_counts = self.log_state = self.log_scalars = None
        if rows > 0:
            C = getattr(model, "class_num", self.cfg.num_classes)
            self.log_counts = torch.zeros((rows, C * C + 3), dtype=torch.float64, device=dev)   # uaps_val_fold's table
            self.log_state = torch.zeros(3, dtype=torch.int32, device=dev)                      # rows, overflow, bad labels
            self.log_scalars = torch.zeros((rows, len(LOG_SCALARS) + self.k), dtype=torch.float64, device=dev)

    # ---- iteration counter (drives the ramp, :279-280) ------------------------------------------------------
    @property
    def iter_num(self) -> int:
        return self._iter

    @iter_num.setter
    def iter_num(self, v: int) -> None:
        self._iter = int(v)
        if self.state is not None:
            self.state.set("iter", int(v))

    def consistency_weights(self):
        c = self.cfg
        return (get_current_consistency_weight(self.iter_num, c.consistency1, c.consistency_rampup, c.iters_per_ramp_epoch),
                get_current_consistency_weight(self.iter_num, c.consistency2, c.consistency_rampup, c.iters_per_ramp_epoch))

    # ---- the three ways to run the iteration -----------------------------------------------------------------
    def step(self, x_l: torch.Tensor, y_l: torch.Tensor, x_u: torch.Tensor,
             mix_w=None, rand_l=None, rand_u=None) -> Dict[str, torch.Tensor]:
        """In captured mode the returned tensors are the graph's static outputs: they are overwritten by the next call
        with the same input shapes (clone what must be kept)."""
        injected = mix_w is not None or rand_l is not None or rand_u is not None
        if self.state is None or injected:
            return self._host_step(x_l, y_l, x_u, mix_w, rand_l, rand_u)
        if not self.cfg.cuda_graph or (self.world > 1 and self.reducer is None):
            # (an NCCL all-reduce inside the iteration is not captured: only the all-kernel iteration is)
            out = self._device_step(x_l, y_l, x_u)
            self._iter += 1
            return out
        key = (tuple(x_l.shape), tuple(y_l.shape), tuple(x_u.shape), x_l.dtype, y_l.dtype)
        cap = self._graphs.get(key)
        if cap is None:
            n = self._warm.get(key, 0)
            if n < max(1, self.cfg.graph_warmup):            # lazy initialisation (module loading, allocator, the weight packer's
                                                             # recording iteration) outside the capture
                self._warm[key] = n + 1
                out = self._device_step(x_l, y_l, x_u)
                self._iter += 1
                return out
            cap = self._capture(key, x_l, y_l, x_u)
        cap.x_l.copy_(x_l, non_blocking=True)
        cap.y_l.copy_(y_l, non_blocking=True)
        cap.x_u.copy_(x_u, non_blocking=True)
        self.optimizer.sync_lr()
        cap.graph.replay()
        self._iter += 1
        return cap.out

    def step_host(self, x_l: torch.Tensor, y_l: torch.Tensor, x_u: torch.Tensor) -> Dict[str, torch.Tensor]:
        """``step`` fed from (pinned) HOST tensors, as a data loader delivers them (UAPS_train.py:160-168 moves each batch with
        ``.cuda()`` and waits for it).  The H2D copies run on a side stream into one of two staging sets, so the copy of
        batch i+1 overlaps the kernels of batch i (the host runs ahead of the device: ``step`` only enqueues work)."""
        dev = self.grads.flat.device
        if not hasattr(self, "_h2d_stream"):
            self._h2d_stream, self._stage, self._stage_free, self._stage_i = torch.cuda.Stream(dev), {}, {}, 0
        main = torch.cuda.current_stream(dev)
        slot = self._stage_i & 1
        self._stage_i += 1
        key = (slot, tuple(x_l.shape), tuple(y_l.shape), tuple(x_u.shape), x_l.dtype, y_l.dtype)
        bufs = self._stage.get(key)
        if bufs is None:
            bufs = tuple(torch.empty(t.shape, dtype=t.dtype, device=dev) for t in (x_l, y_l, x_u))
            self._stage[key] = bufs
        with torch.cuda.stream(self._h2d_stream):
            free = self._stage_free.get(slot)
            if free is not None:
                self._h2d_stream.wait_event(free)             # the iteration that last read this staging set has consumed it
            for d, h in zip(bufs, (x_l, y_l, x_u)):
                d.copy_(h, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(self._h2d_stream)
        main.wait_event(ready)
        out = self.step(*bufs)
        done = torch.cuda.Event()
        done.record(main)
        self._stage_free[slot] = done
        return out

    def _capture(self, key, x_l, y_l, x_u) -> _Captured:
        cap = _Captured()
        cap.x_l, cap.y_l, cap.x_u = torch.empty_like(x_l), torch.empty_like(y_l), torch.empty_like(x_u)
        self.optimizer.sync_lr()
        torch.cuda.synchronize(x_l.device)
        cap.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cap.graph):
            cap.out = self._device_step(cap.x_l, cap.y_l, cap.x_u)
        self._graphs[key] = cap
        return cap

    def _reduce_gradients(self) -> None:
        if self.reducer is None:                 # with a reducer the sum happens inside the optimizer kernel
            self.grads.all_reduce_sum(self.group)

    def _device_step(self, x_l, y_l, x_u) -> Dict[str, torch.Tensor]:
        """The iteration with every per-iteration scalar in device memory: a static launch sequence."""
        st, c = self.state, self.cfg
        self.model.train()
        with pack_scope(), StepContext(x_l.device, state=st, xchg=self.xchg, packer=self.packer):
            st.begin(self.seed_rank, self.seed_shared, self.k, 16, c.consistency1, c.consistency2, c.consistency_rampup,
                     c.iters_per_ramp_epoch, 2 if self.xchg is not None else 0, self.optimizer.betas[0], self.optimizer.betas[1])
            if self.packer.ready:
                self.packer.run()                            # the weights changed in the last optimizer step: re-pack all layers
            out_l = self.model(x_l)                                                              # :177
            out_u = self.model(x_u)                                                              # :185
            sup, tce, tdice, ce_k = uaps_supervised_loss(out_l, y_l, group=self.group, step_state=st)      # :194-218
            loss_u, ps_loss, l_unc, _, _ = uaps_unlabeled_loss(out_u, None, 0.0, 0.0, group=self.group,
                                                               step_state=st)                    # :223-280
            loss = sup + loss_u                                                                  # :282
            if self.log_state is not None:
                self._log_iteration(out_l[0], y_l, (loss, sup, tce, tdice, ps_loss, l_unc), ce_k)   # :295-306
            self.grads.zero()                                                                    # :285
            loss.backward()                                                                      # :287
        self.packer.finalize(x_l.device)                     # (first iteration only: the recorded requests -> device job table)
        self._reduce_gradients()
        # a non-finite loss (an exchange that timed out on a dead peer) must not reach the parameters: the kernel skips
        self.optimizer.step(guard=loss.detach(), use_device_state=True, reducer=self.reducer)    # :292
        return {"loss": loss.detach(), "supervised_loss": sup.detach(), "total_loss_ce": tce.detach(),
                "total_loss_dice": tdice.detach(), "ps_loss": ps_loss.detach(), "l_uncert": l_unc.detach(),
                "loss_ce_k": ce_k}

    def _host_step(self, x_l, y_l, x_u, mix_w, rand_l, rand_u) -> Dict[str, torch.Tensor]:
        self.model.train()
        with pack_scope(), StepContext(x_l.device):          # weights packed once; gradients accumulated in place
            out_l = self.model(x_l) if rand_l is None else self.model(x_l, rand=rand_l)         # :177
            out_u = self.model(x_u) if rand_u is None else self.model(x_u, rand=rand_u)         # :185
            sup, tce, tdice, ce_k = uaps_supervised_loss(out_l, y_l, group=self.group)           # :194-218
            if mix_w is None:
                mix_w = self.rng.dirichlet(np.ones(self.k))                                      # :251
            cw1, cw2 = self.consistency_weights()                                                # :279-280
            loss_u, ps_loss, l_unc, _, _ = uaps_unlabeled_loss(out_u, mix_w, cw1, cw2, group=self.group)  # :223-277
            loss = sup + loss_u                                                                  # :282
            if self.log_state is not None:
                self._log_iteration(out_l[0], y_l, (loss, sup, tce, tdice, ps_loss, l_unc), ce_k)   # :295-306
            self.grads.zero()                                                                    # :285
            loss.backward()                                                                      # :287
        self._reduce_gradients()
        if self.world > 1 and self.reducer is None and not bool(torch.isfinite(loss.detach())):
            # an exchange that timed out yields NaN scalars on every rank: skip the update instead of poisoning the replicas
            warnings.warn("uaps_b200: non-finite loss (loss-sum exchange timed out?); optimizer step skipped")
        elif self.reducer is not None:
            self.optimizer.step(reducer=self.reducer)            # sums the ranks' gradients and updates, one kernel
        else:
            self.optimizer.step()                                                                # :292
        self.iter_num = self._iter + 1
        return {"loss": loss.detach(), "supervised_loss": sup.detach(), "total_loss_ce": tce.detach(),
                "total_loss_dice": tdice.detach(), "ps_loss": ps_loss.detach(), "l_uncert": l_unc.detach(),
                "loss_ce_k": ce_k}

    def skipped_steps(self) -> int:
        """How many optimizer updates the device-side guard has skipped so far (synchronises)."""
        return 0 if self.state is None else int(self.state.read().n_skipped)

    # ---- training log (UAPS_train.py:295-364): per-iteration rows on the device, one read-out per epoch ---------------
    def _log_iteration(self, logits, y_l, scalars, ce_k) -> None:
        """Device work only: the validation head appends the labeled batch's confusion counts of the main output as row
        r = log_state[0] of ``log_counts``; ``uaps_val_scalars`` then copies the iteration's scalars to row r of
        ``log_scalars``."""
        append_row(logits.detach(), y_l, self.log_counts, self.log_state, self._log_ws)
        src, table = [*(t.detach() for t in scalars), *ce_k.detach().unbind()], self.log_scalars
        if len(src) != table.shape[1]:
            raise RuntimeError(f"the training log has {table.shape[1]} scalar columns, the iteration gave {len(src)}")
        with L.on_device(logits.device):
            L.check(L.lib().uaps_val_scalars(L.ptr_array(src), len(src), table.data_ptr(), table.shape[0],
                                             self.log_state.data_ptr(), L.stream_ptr()), "uaps_val_scalars")

    def _require_log(self) -> None:
        if self.log_state is None:
            raise RuntimeError("the training log is off: construct the trainer with UAPSConfig(train_log_rows=n), n > 0")

    @torch.no_grad()
    def log_begin(self) -> None:
        """Start an epoch of the training log: clears its tables (in place: a captured iteration keeps writing to them)."""
        self._require_log()
        self.log_counts.zero_()
        self.log_scalars.zero_()
        self.log_state.zero_()

    def log_result(self) -> Dict[str, object]:
        """The means over the iterations since ``log_begin()`` of what the reference logs per iteration (:295-306) and
        averages per epoch (:316-327): {"loss", "supervised_loss", "total_loss_ce", "total_loss_dice", "ps_loss",
        "l_uncert", "loss_ce_k" (K floats), "pixel_accuracy", "mIoU", "mDice", "iterations"}.  The metrics are those of
        the labeled batch's main-decoder logits, the reference's formulas per iteration, then averaged; under
        torch.distributed each iteration's counts are summed over the ranks first (the whole global batch, as
        DataParallel's gather), while the loss scalars are already global-batch values on every rank.  One all-reduce
        (N > 1) and one host sync.

        These are true means.  The reference runs 59 iterations per epoch but divides its sums by 60 (:159, :316-327);
        its figure is ``value * iterations / 60``.

        Raises when more iterations ran than ``train_log_rows``, when a label was outside [0, C) and not -100, when the
        ranks logged different numbers of iterations, or when no iteration was logged."""
        self._require_log()
        res = finalize(self.log_counts, self.log_state, self.group, scalars=self.log_scalars, errors=_LOG_ERRORS)
        s = res["scalars"]
        out: Dict[str, object] = dict(zip(LOG_SCALARS, s))
        out["loss_ce_k"] = s[len(LOG_SCALARS):]
        out.update(pixel_accuracy=res["pixel_accuracy"], mIoU=res["mIoU"], mDice=res["mDice"], iterations=res["batches"])
        return out
