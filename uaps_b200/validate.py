"""Per-epoch validation on the device: the reference's validation pass (UAPS_train.py:367-402) as one CUDA graph per
input shape and one host sync per epoch (DESIGN.md f6).

    val = Validator(model)              # once
    val.begin()                         # every epoch, after training: snapshot of the current weights / running statistics
    for x, y in val_loader:
        val.update(x, y)                # main decoder's logits + the validation head, appended as one row of a device table
    res = val.result()                  # {"val_loss", "ce", "pixel_accuracy", "mIoU", "mDice", "batches"}
    scheduler.step(res["mDice"])        # :402

Per batch the reference computes CrossEntropyLoss()(logits, y) (:383, torch's ignore_index -100), pixel accuracy, mIoU
and mDice (utilities/metrics.py) and val_loss = CE + (1 - mDice) (:385), and averages each over the epoch's batches
(:395-400).  Here the batch's confusion matrix and CE sum are one row of an epoch table filled by ``uaps_val_counts`` +
``uaps_val_fold``; ``result()`` applies the reference's formulas to every row and averages the rows.  Under
torch.distributed (one process per GPU, each holding a shard of every batch) the tables are summed once, so row i holds
the counts of the WHOLE batch i -- what DataParallel's gather to GPU 0 gives the reference.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.distributed as dist

from . import _lib as L
from .conv import PackedConv
from .metrics import metrics_from_confusion
from .unet import _check_hw

IGNORE_INDEX = -100


def _world(group):
    if group is None or not dist.is_available() or not dist.is_initialized():
        return 1, 0
    world = dist.get_world_size(group)
    return world, (dist.get_rank(group) if world > 1 else 0)


VAL_ERRORS = {"ranks": "the ranks validated different numbers of batches",
              "overflow": "more validation batches than max_batches since begin()",
              "empty": "no validation batch since begin()"}


def finalize(table: torch.Tensor, state: torch.Tensor, group=None, scalars: Optional[torch.Tensor] = None,
             errors: Dict[str, str] = VAL_ERRORS) -> Dict[str, float]:
    """The epoch's result from the table ``uaps_val_fold`` fills: fp64 [max_batches, C*C + 3] rows of C*C confusion counts
    | CE sum | non-ignored pixels | pixels, and ``state`` = (rows written, overflow flag, bad labels).  Plain torch ops on
    whatever device the tensors live on; the only host sync is the final read-out.  With a process group of N > 1 ranks
    the table and the state are summed over the ranks in ONE all-reduce first; every rank must have written the same
    number of rows.

    ``scalars``: an optional [max_batches, S] table row-aligned with ``table`` (``uaps_val_scalars``); the result then also
    holds ``"scalars"``, its S column means over the written rows, read out in the same sync.  These are this rank's own
    values and are not summed over the ranks.  ``errors``: the messages raised for mismatched row counts, overflow and an
    empty table."""
    world, rank = _world(group)
    C = int(round((table.shape[1] - 3) ** 0.5))
    if C * C + 3 != table.shape[1]:
        raise ValueError("table rows must hold C*C + 3 values")
    if scalars is not None and (scalars.dim() != 2 or scalars.shape[0] != table.shape[0]):
        raise ValueError("the scalar table must have one row per row of the counts table")
    ext = torch.zeros(world + 2, dtype=torch.float64, device=table.device)
    ext[rank] = state[0]                                      # each rank's row count in its own slot: compared after the sum
    ext[world:] = state[1:3]
    buf = torch.cat([table.reshape(-1).double(), ext])
    if world > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    tab, ext = buf[:table.numel()].view(table.shape), buf[table.numel():]
    n = ext[0]
    acc, miou, mdice = metrics_from_confusion(tab[:, :C * C].view(-1, C, C), n_pixels=tab[:, C * C + 2])
    ce = tab[:, C * C] / tab[:, C * C + 1]                    # 0 / 0 = NaN when every pixel is ignored, as torch
    per_row = torch.stack([ce + (1 - mdice), ce, acc, miou, mdice], 1)
    written = (torch.arange(table.shape[0], device=table.device) < n)[:, None]
    zero = torch.zeros((), dtype=torch.float64, device=table.device)
    if scalars is not None:
        per_row = torch.cat([per_row, scalars.double()], 1)
    means = torch.where(written, per_row, zero).sum(0) / n.clamp(min=1)
    host = torch.cat([means, ext]).tolist()                   # the one host sync
    m = means.numel()
    rows, overflow, bad = [int(v) for v in host[m:m + world]], host[m + world], host[m + world + 1]
    if len(set(rows)) != 1:
        raise RuntimeError(f"{errors['ranks']}: {rows}")
    if overflow:
        raise RuntimeError(errors["overflow"])
    if bad:
        raise RuntimeError(f"{int(bad)} labels outside [0, C) that are not the ignore index {IGNORE_INDEX}")
    if rows[0] == 0:
        raise RuntimeError(errors["empty"])
    res = {"val_loss": host[0], "ce": host[1], "pixel_accuracy": host[2], "mIoU": host[3], "mDice": host[4],
           "batches": rows[0]}
    if scalars is not None:
        res["scalars"] = host[5:m]
    return res


def append_row(logits: torch.Tensor, y: torch.Tensor, table: torch.Tensor, state: torch.Tensor,
               workspaces: Dict[tuple, torch.Tensor]) -> None:
    """The validation head on one batch: fp32 logits [B, C, H, W] and int64 labels ([B, H, W] or [B, H*W]) become the
    next row of ``table`` (``uaps_val_counts`` + ``uaps_val_fold``).  ``workspaces``: the caller's cache of head
    workspaces per (B, H*W); a missing one is allocated here, so call once eagerly per shape before a graph capture."""
    B, C, H, W = logits.shape
    if table.shape[1] != C * C + 3:
        raise ValueError(f"table rows hold {table.shape[1]} values, the logits' {C} classes need {C * C + 3}")
    logits, y = logits.contiguous(), y.reshape(B, H * W).contiguous()
    lib = L.lib()
    ws = workspaces.get((B, H * W))
    if ws is None:
        ws = torch.empty(lib.uaps_val_workspace_bytes(C, B, H * W), dtype=torch.uint8, device=logits.device)
        workspaces[(B, H * W)] = ws
    with L.on_device(logits.device):
        L.check(lib.uaps_val_counts(logits.data_ptr(), y.data_ptr(), B, C, H * W, ws.data_ptr(), ws.numel(),
                                    L.stream_ptr()), "uaps_val_counts")
        L.check(lib.uaps_val_fold(ws.data_ptr(), ws.numel(), B, C, H * W, table.data_ptr(), table.shape[0],
                                  state.data_ptr(), L.stream_ptr()), "uaps_val_fold")


def _owned_layer(w, b, cin_split=None):
    return PackedConv(w, None if b is None else b.detach().float().clone(), cin_split=cin_split)


def _layers(plan):
    """The PackedConv objects of an (enc, dec, out) plan in the order ``UNet_UAPS._main_plan`` builds them."""
    enc, dec, out = plan
    return [pc for blk in enc for pc in blk] + [pc for up in dec for pc in up] + [out]


class Validator:
    """Validation of a ``UNet_UAPS`` with BatchNorm's running statistics (the reference's ``model.eval()``), whatever mode
    the model is in.  ``max_batches``: rows of the epoch table (batches per epoch).  ``group``: the process group whose
    ranks each hold a shard of every validation batch (default: WORLD under torchrun, as ``UAPSTrainer``)."""

    def __init__(self, model, max_batches: int = 4096, group=None):
        if group is None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            group = dist.group.WORLD
        dev = next(model.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("uaps_b200 kernels run on CUDA tensors only (no CPU fallback)")
        if max_batches < 1:
            raise ValueError("max_batches must be positive")
        self.model, self.group, self.max_batches = model, group, int(max_batches)
        C = model.class_num
        self.table = torch.zeros((self.max_batches, C * C + 3), dtype=torch.float64, device=dev)
        self.state = torch.zeros(3, dtype=torch.int32, device=dev)
        self.captures = 0                 # CUDA graphs captured so far (one per input shape, kept for the validator's life)
        self._plan = None
        self._begun = False
        self._graphs, self._seen, self._ws = {}, set(), {}

    @torch.no_grad()
    def begin(self) -> None:
        """Start an epoch: fold the model's CURRENT weights and BatchNorm running statistics into the validator's own
        packed layers (in place, so the captured graphs stay valid) and clear the table."""
        if self.model.compute == "bf16":
            if self._plan is None:
                self._plan = self.model._main_plan(make=_owned_layer)
            else:
                layers = iter(_layers(self._plan))
                self.model._main_plan(make=lambda w, b, cin_split=None: next(layers).repack(w, b))
                assert next(layers, None) is None
        self.table.zero_()
        self.state.zero_()
        self._begun = True

    @torch.no_grad()
    def update(self, x: torch.Tensor, y: torch.Tensor) -> None:
        """One validation batch: x [B, in_chns, H, W], y integer labels [B, H, W] or [B, 1, H, W] (-100 = ignored).
        Enqueues device work only.  On the bf16 path the first batch of an input shape runs eagerly and the next one
        captures the forward + head into a CUDA graph that every later batch of that shape replays."""
        if not self._begun:
            raise RuntimeError("call begin() before update()")
        L.require_cuda(x, y)
        _check_hw(x)
        B, _, H, W = x.shape
        if tuple(y.shape) not in ((B, H, W), (B, 1, H, W)):
            raise ValueError(f"labels must be [B, H, W] or [B, 1, H, W] for inputs {tuple(x.shape)}, got {tuple(y.shape)}")
        if y.dtype.is_floating_point or y.dtype == torch.bool:
            raise ValueError("labels must be an integer tensor")
        y = y.reshape(B, H, W)
        if self.model.compute != "bf16":
            was = self.model.training
            self.model.eval()
            try:
                logits = self.model.predict(x)
            finally:
                self.model.train(was)
            self._head(logits, y.long().contiguous())
            return
        key = (tuple(x.shape), x.dtype, x.device.index)
        entry = self._graphs.get(key)
        if entry is None:
            if key not in self._seen:
                self._seen.add(key)
                self._run(x, y.long().contiguous())
                return
            entry = self._capture(key, x, y)
        static_x, static_y, graph = entry
        static_x.copy_(x)
        static_y.copy_(y)
        graph.replay()

    def result(self) -> Dict[str, float]:
        """{"val_loss", "ce", "pixel_accuracy", "mIoU", "mDice", "batches"} of the batches since ``begin()``: one
        all-reduce (N > 1) and one host sync.  Raises when a label was outside [0, C) and not -100, when more than
        ``max_batches`` batches were given, or when the ranks gave different numbers of batches."""
        return finalize(self.table, self.state, self.group)

    # ---- internals ---------------------------------------------------------------------------------------------------
    def _run(self, x, y):
        enc, dec, out = self._plan
        self._head(self.model._decode_folded(self.model._encode_folded(x, enc), dec, out), y)

    def _capture(self, key, x, y):
        static_x = torch.empty_like(x)
        static_y = torch.empty(y.shape, dtype=torch.int64, device=x.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self._run(static_x, static_y)
        self.captures += 1
        self._graphs[key] = (static_x, static_y, graph)
        return self._graphs[key]

    def _head(self, logits: torch.Tensor, y: torch.Tensor) -> None:
        append_row(logits, y, self.table, self.state, self._ws)
