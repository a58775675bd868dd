"""Host side of the training log (no GPU needed): ``validate.finalize`` with a row-aligned scalar table on hand-built
tables, the trainer's read-out and error messages on a CPU trainer, the reduction over two gloo ranks (counts summed,
scalars this rank's own), and the C ABI of ``uaps_val_scalars`` (export, argument checks before any launch)."""
import ctypes
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F


def _row(logits, mask, C):
    """The row uaps_val_fold writes, restated on the CPU (as test_validate_cpu.py)."""
    pred = torch.argmax(torch.softmax(logits, 1), 1)
    keep = (mask >= 0) & (mask < C)
    conf = torch.bincount((mask[keep] * C + pred[keep]).view(-1), minlength=C * C).double()
    ce = F.cross_entropy(logits.double(), mask, reduction="sum")
    return torch.cat([conf, torch.stack([ce, keep.sum().double(), torch.tensor(float(mask.numel()), dtype=torch.float64)])])


def _batch(g, B, C, H, W):
    return torch.randn(B, C, H, W, generator=g) * 2, torch.randint(0, C, (B, H, W), generator=g)


def _scalar_rows(g, n, S):
    """Per-iteration loss scalars as uaps_val_scalars stores them: fp32 values widened to fp64."""
    return (torch.rand(n, S, generator=g) * 3).double()


def _tables(rows, scalars, max_rows=8):
    t = torch.zeros(max_rows, rows[0].numel(), dtype=torch.float64)
    s = torch.zeros(max_rows, scalars.shape[1], dtype=torch.float64)
    for i, r in enumerate(rows):
        t[i], s[i] = r, scalars[i]
    return t, torch.tensor([len(rows), 0, 0], dtype=torch.int32), s


def test_finalize_averages_the_scalar_columns_and_keeps_the_metrics():
    from uaps_b200.metrics import metrics_from_confusion
    from uaps_b200.validate import finalize
    g = torch.Generator().manual_seed(21)
    C, S = 4, 10
    batches = [_batch(g, 2, C, 16, 24) for _ in range(3)]
    rows = [_row(z, y, C) for z, y in batches]
    sc = _scalar_rows(g, 3, S)
    table, state, scalars = _tables(rows, sc)
    scalars[3:] = 7.0                                         # rows past the written ones must not count
    res = finalize(table, state, scalars=scalars)
    assert res["scalars"] == pytest.approx(sc.mean(0).tolist(), rel=1e-12) and len(res["scalars"]) == S
    without = finalize(table, state)
    for k in ("val_loss", "ce", "pixel_accuracy", "mIoU", "mDice", "batches"):
        assert res[k] == without[k], k
    want = [metrics_from_confusion(r[:C * C].view(C, C), n_pixels=y.numel()) for r, (_, y) in zip(rows, batches)]
    for i, k in enumerate(("pixel_accuracy", "mIoU", "mDice")):
        assert res[k] == pytest.approx(sum(float(w[i]) for w in want) / 3, rel=1e-12), k
    with pytest.raises(ValueError, match="one row per row"):
        finalize(table, state, scalars=scalars[:5])


def _cpu_trainer(rows, C=4, n_aux=3):
    from uaps_b200.train import UAPSConfig, UAPSTrainer
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(0)
    return UAPSTrainer(UNet_UAPS(3, C, n_aux=n_aux), UAPSConfig(num_classes=C, optimizer="torch", train_log_rows=rows))


def test_log_result_names_the_columns_and_reports_the_mean():
    from uaps_b200.train import LOG_SCALARS
    g = torch.Generator().manual_seed(22)
    C, n_aux = 2, 4
    tr = _cpu_trainer(6, C=C, n_aux=n_aux)
    K = n_aux + 1
    assert tr.log_counts.shape == (6, C * C + 3) and tr.log_scalars.shape == (6, len(LOG_SCALARS) + K)
    batches = [_batch(g, 2, C, 8, 8) for _ in range(4)]
    sc = _scalar_rows(g, 4, len(LOG_SCALARS) + K)
    for i, (z, y) in enumerate(batches):
        tr.log_counts[i], tr.log_scalars[i] = _row(z, y, C), sc[i]
    tr.log_state[0] = 4
    res = tr.log_result()
    assert set(res) == {*LOG_SCALARS, "loss_ce_k", "pixel_accuracy", "mIoU", "mDice", "iterations"}
    mean = sc.mean(0).tolist()
    for j, k in enumerate(LOG_SCALARS):
        assert res[k] == pytest.approx(mean[j], rel=1e-12), k
    assert res["loss_ce_k"] == pytest.approx(mean[len(LOG_SCALARS):], rel=1e-12) and len(res["loss_ce_k"]) == K
    assert res["iterations"] == 4
    # the reference divides its sums by 60 over 59 iterations: mean * iterations / 60 is its figure
    assert res["loss"] * res["iterations"] / 60 == pytest.approx(sc[:, 0].sum().item() / 60, rel=1e-12)
    tr.log_begin()
    assert tr.log_counts.abs().sum() == 0 and tr.log_scalars.abs().sum() == 0 and tr.log_state.tolist() == [0, 0, 0]


def test_log_result_raises_on_flags():
    g = torch.Generator().manual_seed(23)
    tr = _cpu_trainer(2)
    tr.log_counts[0] = _row(*_batch(g, 1, 4, 8, 8), 4)
    for state, msg in (([1, 1, 0], "more training iterations than UAPSConfig.train_log_rows"),
                       ([1, 0, 5], "5 labels outside"), ([0, 0, 0], "no training iteration logged")):
        tr.log_state.copy_(torch.tensor(state, dtype=torch.int32))
        with pytest.raises(RuntimeError, match=msg):
            tr.log_result()


def test_log_off_refuses_the_epoch_api():
    tr = _cpu_trainer(0)
    assert tr.log_counts is None and tr.log_scalars is None and tr.log_state is None
    for fn in (tr.log_begin, tr.log_result):
        with pytest.raises(RuntimeError, match="training log is off"):
            fn()
    with pytest.raises(ValueError, match="train_log_rows"):
        _cpu_trainer(-1)


# ---- two gloo ranks, each holding half of every labeled batch ---------------------------------------------------------
C2, NB, B2, S2 = 4, 3, 4, 10


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _epoch():
    g = torch.Generator().manual_seed(31)
    return [_batch(g, B2, C2, 16, 16) for _ in range(NB)], _scalar_rows(g, NB, S2)


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from uaps_b200.train import _LOG_ERRORS
        from uaps_b200.validate import finalize
        batches, sc = _epoch()
        per = B2 // world
        rows = [_row(z[rank * per:(rank + 1) * per], y[rank * per:(rank + 1) * per], C2) for z, y in batches]
        table, state, scalars = _tables(rows, sc)
        ret[rank] = finalize(table, state, dist.group.WORLD, scalars=scalars, errors=_LOG_ERRORS)
        try:                                                   # rank 1 logged one iteration less: every rank must refuse
            table, state, scalars = _tables(rows if rank == 0 else rows[:-1], sc)
            finalize(table, state, dist.group.WORLD, scalars=scalars, errors=_LOG_ERRORS)
            ret[rank + world] = "no error"
        except RuntimeError as e:
            ret[rank + world] = str(e)
    finally:
        dist.destroy_process_group()


def test_two_ranks_sum_the_counts_and_keep_the_scalars():
    from uaps_b200.validate import finalize
    world, port = 2, _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
    batches, sc = _epoch()
    table, state, scalars = _tables([_row(z, y, C2) for z, y in batches], sc)
    want = finalize(table, state, scalars=scalars)
    for rank in range(world):
        got = ret[rank]
        assert got["batches"] == want["batches"] == NB
        for k in ("pixel_accuracy", "mIoU", "mDice"):
            assert got[k] == pytest.approx(want[k], rel=1e-12), k
        assert got["scalars"] == want["scalars"]                # not summed: identical on every rank, bit for bit
        assert "different numbers of training iterations" in ret[rank + world]


# ---- the C ABI --------------------------------------------------------------------------------------------------------
def test_val_scalars_abi_export_and_host_checks():
    from uaps_b200 import _lib as L
    handle = ctypes.CDLL(L.LIB_PATH)
    assert hasattr(handle, "uaps_val_scalars") and "uaps_val_scalars" in L.exported_symbols()
    lib = L.lib()
    fake, odd = 4096, 4098                                   # never dereferenced: every call fails its checks first
    src = (ctypes.c_void_p * 17)(*([fake] * 17))
    assert lib.uaps_val_scalars(None, 4, fake, 8, fake, None) == -1
    assert lib.uaps_val_scalars(src, 4, None, 8, fake, None) == -1
    assert lib.uaps_val_scalars(src, 4, fake, 8, None, None) == -1
    assert lib.uaps_val_scalars(src, 4, fake, -1, fake, None) == -1
    assert lib.uaps_val_scalars(src, 0, fake, 8, fake, None) == -2
    assert lib.uaps_val_scalars(src, 17, fake, 8, fake, None) == -2
    assert lib.uaps_val_scalars(src, 4, odd, 8, fake, None) == -3
    assert lib.uaps_val_scalars(src, 4, fake, 8, fake + 2, None) == -3
    bad = (ctypes.c_void_p * 4)(fake, fake, None, fake)
    assert lib.uaps_val_scalars(bad, 4, fake, 8, fake, None) == -1
    bad[2] = odd
    assert lib.uaps_val_scalars(bad, 4, fake, 8, fake, None) == -3
