"""Host side of the validation path (no GPU needed): the epoch finalize of ``uaps_b200.validate`` on CPU tensors against
``metrics_from_confusion`` and the reference's own metric outputs, its reduction over two gloo ranks, its error flags,
and the C ABI of the validation head (exports, workspace size, argument checks before any launch)."""
import ctypes
import math
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F


def _row(logits, mask, C):
    """The table row uaps_val_fold writes, restated on the CPU: confusion (label, argmax softmax) over the labels in
    [0, C) | CE sum | non-ignored pixels | pixels."""
    pred = torch.argmax(torch.softmax(logits, 1), 1)
    keep = (mask >= 0) & (mask < C)
    conf = torch.bincount((mask[keep] * C + pred[keep]).view(-1), minlength=C * C).double()
    ce = F.cross_entropy(logits.double(), mask, reduction="sum")          # ignore_index -100
    return torch.cat([conf, torch.stack([ce, keep.sum().double(), torch.tensor(float(mask.numel()), dtype=torch.float64)])])


def _table(rows, max_batches=8):
    t = torch.zeros(max_batches, rows[0].numel(), dtype=torch.float64)
    for i, r in enumerate(rows):
        t[i] = r
    return t, torch.tensor([len(rows), 0, 0], dtype=torch.int32)


def _batch(g, B, C, H, W, absent=None, ignore=0.0):
    logits = torch.randn(B, C, H, W, generator=g) * 2
    mask = torch.randint(0, C, (B, H, W), generator=g)
    if absent is not None:
        mask[mask == absent] = 0
    if ignore:
        mask[torch.rand(B, H, W, generator=g) < ignore] = -100
    return logits, mask


def test_finalize_applies_the_reference_formulas_per_row_then_averages():
    from uaps_b200.metrics import metrics_from_confusion
    from uaps_b200.validate import finalize
    g = torch.Generator().manual_seed(3)
    C = 4
    batches = [_batch(g, 2, C, 16, 24), _batch(g, 3, C, 16, 16, absent=2, ignore=0.1), _batch(g, 1, C, 32, 16, absent=3)]
    rows = [_row(z, y, C) for z, y in batches]
    res = finalize(*_table(rows))
    want = []
    for (z, y), r in zip(batches, rows):
        acc, miou, mdice = (float(v) for v in metrics_from_confusion(r[:C * C].view(C, C), n_pixels=y.numel()))
        ce = F.cross_entropy(z.double(), y).item()                         # mean over the non-ignored pixels
        assert r[C * C].item() / r[C * C + 1].item() == pytest.approx(ce, rel=1e-12)
        want.append((ce + 1 - mdice, ce, acc, miou, mdice))
    for i, k in enumerate(("val_loss", "ce", "pixel_accuracy", "mIoU", "mDice")):
        assert res[k] == pytest.approx(sum(w[i] for w in want) / len(want), rel=1e-12), k
    assert res["batches"] == 3


def test_finalize_nan_rules():
    """A batch without any foreground label has no mIoU / mDice (np.nanmean of nothing), a batch whose pixels are all
    ignored has no CE (torch: 0 / 0): either makes the epoch mean NaN, as the reference's running average."""
    from uaps_b200.validate import finalize
    g = torch.Generator().manual_seed(4)
    z, y = _batch(g, 2, 3, 16, 16)
    good = _row(z, y, 3)
    res = finalize(*_table([good, _row(z, torch.zeros_like(y), 3)]))
    assert math.isnan(res["mIoU"]) and math.isnan(res["mDice"]) and math.isnan(res["val_loss"])
    assert not math.isnan(res["ce"]) and not math.isnan(res["pixel_accuracy"])
    res = finalize(*_table([good, _row(z, torch.full_like(y, -100), 3)]))
    assert math.isnan(res["ce"]) and math.isnan(res["val_loss"])
    assert res["pixel_accuracy"] == pytest.approx(finalize(*_table([good]))["pixel_accuracy"] / 2, rel=1e-12)


def test_finalize_matches_reference_golden():
    """tests/golden/metrics.npz holds what the reference's own utilities/metrics.py returned for these logits / masks."""
    from conftest import load_cases
    from uaps_b200.validate import finalize
    for name, c in load_cases("metrics.npz").items():
        z, y, C = torch.from_numpy(c["logits"]), torch.from_numpy(c["mask"]), int(c["n_classes"])
        res = finalize(*_table([_row(z, y, C)], max_batches=3))
        assert res["pixel_accuracy"] == pytest.approx(float(c["pixel_accuracy"]), rel=1e-12), name
        assert res["mIoU"] == pytest.approx(float(c["mIoU"]), rel=1e-9), name
        assert res["mDice"] == pytest.approx(float(c["mDice"]), rel=1e-9), name
        ce = F.cross_entropy(z.double(), y).item()
        assert res["ce"] == pytest.approx(ce, rel=1e-12), name
        assert res["val_loss"] == pytest.approx(ce + 1 - float(c["mDice"]), rel=1e-9), name


def test_finalize_raises_on_flags():
    from uaps_b200.validate import finalize
    g = torch.Generator().manual_seed(5)
    table, state = _table([_row(*_batch(g, 1, 2, 16, 16), 2)])
    for bad_state, msg in (([1, 1, 0], "max_batches"), ([1, 0, 3], "outside"), ([0, 0, 0], "no validation batch")):
        with pytest.raises(RuntimeError, match=msg):
            finalize(table, torch.tensor(bad_state, dtype=torch.int32))
    with pytest.raises(ValueError):
        finalize(torch.zeros(4, 10, dtype=torch.float64), state)


# ---- two gloo ranks, each holding half of every batch ----------------------------------------------------------------
C2, NB, B2 = 4, 3, 4


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _epoch():
    g = torch.Generator().manual_seed(11)
    return [_batch(g, B2, C2, 16, 16, absent=(2 if i == 1 else None), ignore=0.05) for i in range(NB)]


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from uaps_b200.validate import finalize
        per = B2 // world
        rows = [_row(z[rank * per:(rank + 1) * per], y[rank * per:(rank + 1) * per], C2) for z, y in _epoch()]
        ret[rank] = finalize(*_table(rows), group=dist.group.WORLD)
        try:                                                   # rank 1 misses the last batch: every rank must refuse
            finalize(*_table(rows if rank == 0 else rows[:-1]), group=dist.group.WORLD)
            ret[rank + world] = "no error"
        except RuntimeError as e:
            ret[rank + world] = str(e)
    finally:
        dist.destroy_process_group()


def test_two_ranks_reduce_to_the_whole_batch_result():
    from uaps_b200.validate import finalize
    world, port = 2, _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    want = finalize(*_table([_row(z, y, C2) for z, y in _epoch()]))
    for rank in range(world):
        got = ret[rank]
        assert got["batches"] == want["batches"] == NB
        for k in ("val_loss", "ce", "pixel_accuracy", "mIoU", "mDice"):
            assert got[k] == pytest.approx(want[k], rel=1e-12), k
        assert "different numbers of batches" in ret[rank + world]


# ---- the C ABI --------------------------------------------------------------------------------------------------------
def test_val_abi_exports_and_host_checks():
    from uaps_b200 import _lib as L
    handle = ctypes.CDLL(L.LIB_PATH)
    for name in ("uaps_val_workspace_bytes", "uaps_val_counts", "uaps_val_fold"):
        assert hasattr(handle, name) and name in L.exported_symbols()
    lib = L.lib()
    # 64 x 256^2: 2048-pixel chunks, 32 per image -> 2048 blocks of (one double + C*C + 2 words)
    assert lib.uaps_val_workspace_bytes(4, 64, 65536) == 2048 * 8 + 18 * 2048 * 4
    assert lib.uaps_val_workspace_bytes(2, 1, 63) == 8 + 6 * 4
    for C, B, HW in ((1, 1, 64), (9, 1, 64), (4, 0, 64), (4, 1, 0), (4, 65536, 16), (4, 4096, 1 << 20)):
        assert lib.uaps_val_workspace_bytes(C, B, HW) == 0
    fake, odd = ctypes.c_void_p(4096), ctypes.c_void_p(4098)    # never dereferenced: every call fails its checks first
    need = lib.uaps_val_workspace_bytes(4, 1, 64)
    assert lib.uaps_val_counts(None, fake, 1, 4, 64, fake, need, None) == -1
    assert lib.uaps_val_counts(fake, fake, 1, 4, 64, None, need, None) == -1
    assert lib.uaps_val_counts(fake, fake, 1, 9, 64, fake, need, None) == -2
    assert lib.uaps_val_counts(odd, fake, 1, 4, 64, fake, need, None) == -3
    assert lib.uaps_val_counts(fake, odd, 1, 4, 64, fake, need, None) == -3
    assert lib.uaps_val_counts(fake, fake, 1, 4, 64, fake, need - 1, None) == -1
    assert lib.uaps_val_fold(fake, need, 1, 4, 64, None, 8, fake, None) == -1
    assert lib.uaps_val_fold(fake, need, 1, 4, 64, fake, -1, fake, None) == -1
    assert lib.uaps_val_fold(fake, need, 1, 4, 64, fake, 8, odd, None) == -3
    assert lib.uaps_val_fold(fake, need - 1, 1, 4, 64, fake, 8, fake, None) == -1


def test_validator_refuses_a_cpu_model():
    from uaps_b200.unet import UNet_UAPS
    from uaps_b200.validate import Validator
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        Validator(UNet_UAPS(3, 4))
