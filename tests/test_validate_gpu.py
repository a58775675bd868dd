"""The validation path on the GPU: the head (uaps_val_counts + uaps_val_fold) against uaps_confusion, torch's argmax and
fp64 cross-entropy; determinism, graph replay and overflow; and ``Validator`` end to end between training epochs against
predict + ce_loss + MetricAccumulator."""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _head(logits, labels, max_batches=4, table=None, state=None):
    """One counts + fold launch pair; returns (table, state) (synchronised)."""
    from uaps_b200 import _lib as L
    lib = L.lib()
    B, C, H, W = logits.shape
    if table is None:
        table = torch.zeros(max_batches, C * C + 3, dtype=torch.float64, device=DEV)
        state = torch.zeros(3, dtype=torch.int32, device=DEV)
    ws = torch.empty(lib.uaps_val_workspace_bytes(C, B, H * W), dtype=torch.uint8, device=DEV)
    ws.fill_(0xAB)                                           # no zero-fill needed: every partial is written before it is read
    y = labels.reshape(B, H * W).contiguous()
    L.check(lib.uaps_val_counts(logits.data_ptr(), y.data_ptr(), B, C, H * W, ws.data_ptr(), ws.numel(), L.stream_ptr()),
            "uaps_val_counts")
    L.check(lib.uaps_val_fold(ws.data_ptr(), ws.numel(), B, C, H * W, table.data_ptr(), table.shape[0], state.data_ptr(),
                              L.stream_ptr()), "uaps_val_fold")
    torch.cuda.synchronize()
    return table, state


def _near_tie_logits(g, B, C, H, W):
    z = torch.randn(B, C, H, W, generator=g, device=DEV) * 2
    pick = torch.rand(B, H, W, generator=g, device=DEV)
    for c in range(1, C):                                    # duplicated class planes (exact ties) and 1-ulp neighbours
        z[:, c] = torch.where(pick < 0.1, z[:, 0], z[:, c])
        z[:, c] = torch.where((pick >= 0.1) & (pick < 0.2), torch.nextafter(z[:, 0], z[:, 0] + 1), z[:, c])
    return z


SHAPES = [(1, 7, 9), (3, 6, 5), (3, 33, 34), (64, 16, 16), (3, 32, 48)]   # HW odd, HW % 2 only (x2), vectorised (x2)


@pytest.mark.parametrize("C", range(2, 9))
@pytest.mark.parametrize("B,H,W", SHAPES)
def test_counts_equal_uaps_confusion_and_torch_argmax(C, B, H, W):
    from uaps_b200.metrics import confusion
    g = torch.Generator(device=DEV).manual_seed(100 * C + H)
    z = _near_tie_logits(g, B, C, H, W)
    y = torch.randint(0, C, (B, H, W), generator=g, device=DEV)
    table, state = _head(z, y)
    got = table[0, :C * C].view(C, C)
    assert torch.equal(got.long(), confusion(z, y))
    pred = torch.argmax(torch.softmax(z, 1), 1)
    want = torch.bincount((y * C + pred).view(-1), minlength=C * C).view(C, C)
    assert torch.equal(got.long(), want)
    assert table[0, C * C + 1].item() == table[0, C * C + 2].item() == B * H * W
    assert state.tolist() == [1, 0, 0] and table[1:].abs().sum().item() == 0


@pytest.mark.parametrize("C", [2, 4, 7])
@pytest.mark.parametrize("B,H,W", [(1, 7, 9), (3, 6, 5), (64, 16, 16)])
def test_ce_sum_matches_fp64_cross_entropy_with_ignored_pixels(C, B, H, W):
    g = torch.Generator(device=DEV).manual_seed(C + B)
    z = torch.randn(B, C, H, W, generator=g, device=DEV) * 3
    y = torch.randint(0, C, (B, H, W), generator=g, device=DEV)
    y[torch.rand(B, H, W, generator=g, device=DEV) < 0.2] = -100
    table, state = _head(z, y)
    want = F.cross_entropy(z.double(), y, reduction="sum").item()
    assert table[0, C * C].item() == pytest.approx(want, rel=1e-6)
    keep = y != -100
    assert table[0, C * C + 1].item() == keep.sum().item() and table[0, C * C + 2].item() == y.numel()
    pred = torch.argmax(torch.softmax(z, 1), 1)
    want_conf = torch.bincount((y[keep] * C + pred[keep]), minlength=C * C)
    assert torch.equal(table[0, :C * C].long(), want_conf) and state.tolist() == [1, 0, 0]


def test_all_ignored_batch_gives_nan_ce_and_bad_labels_raise():
    from uaps_b200.validate import finalize
    z = torch.randn(2, 4, 16, 16, device=DEV)
    y = torch.full((2, 16, 16), -100, dtype=torch.int64, device=DEV)
    res = finalize(*_head(z, y))
    assert torch.isnan(F.cross_entropy(z, y)).item()
    assert res["ce"] != res["ce"] and res["pixel_accuracy"] == 0.0
    for bad in (4, -1):
        y2 = torch.randint(0, 4, (2, 16, 16), device=DEV)
        y2[1, 3, 5] = bad
        y2[0, 0, 0] = bad
        table, state = _head(z, y2)
        assert state.tolist() == [1, 0, 2]
        assert table[0, 17].item() == y2.numel() - 2
        with pytest.raises(RuntimeError, match="outside"):
            finalize(table, state)


def test_rows_are_bitwise_reproducible():
    g = torch.Generator(device=DEV).manual_seed(9)
    z = torch.randn(16, 4, 256, 256, generator=g, device=DEV) * 4
    y = torch.randint(0, 4, (16, 256, 256), generator=g, device=DEV)
    a, _ = _head(z, y)
    b, _ = _head(z, y)
    assert torch.equal(a, b)
    assert a[0, 16].item() == pytest.approx(F.cross_entropy(z.double(), y, reduction="sum").item(), rel=1e-6)


def _small_model(seed=0, C=4, compute="bf16"):
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(seed)
    return UNet_UAPS(3, C, compute=compute).to(DEV)


def _val_data(n, B=4, H=64, W=64, C=4, seed=1):
    g = torch.Generator(device=DEV).manual_seed(seed)
    xs = [torch.randn(B, 3, H, W, generator=g, device=DEV) for _ in range(n)]
    ys = [((x[:, 0] > 0).long() + 2 * (x[:, 1] > 0.5).long()).clamp(max=C - 1) for x in xs]
    return xs, ys


def test_graph_replays_fill_consecutive_rows_like_eager_calls_and_overflow_raises():
    from uaps_b200.validate import Validator
    m = _small_model()
    xs, ys = _val_data(5)
    val = Validator(m, max_batches=8)
    val.begin()
    for x, y in zip(xs, ys):
        val.update(x, y.unsqueeze(1))                       # [B,1,H,W] labels, as the reference's loaders give them
    assert val.captures == 1
    eager = Validator(m, max_batches=8)
    eager.begin()
    for x, y in zip(xs, ys):
        eager._run(x, y)                                    # the same forward + head, launched one by one
    torch.cuda.synchronize()
    assert val.state.tolist() == eager.state.tolist() == [5, 0, 0]
    assert torch.equal(val.table, eager.table) and val.table[4].abs().sum() > 0 and val.table[5:].abs().sum() == 0
    val.begin()                                             # a new epoch: table cleared, same graph
    for x, y in zip(xs[:3], ys[:3]):
        val.update(x, y)
    torch.cuda.synchronize()
    assert val.captures == 1 and torch.equal(val.table[:3], eager.table[:3]) and val.table[3:].abs().sum() == 0
    small = Validator(m, max_batches=2)
    small.begin()
    for x, y in zip(xs[:3], ys[:3]):
        small.update(x, y)
    torch.cuda.synchronize()
    assert small.state.tolist() == [2, 1, 0]
    with pytest.raises(RuntimeError, match="max_batches"):
        small.result()


def _reference_epoch(model_state, xs, ys, C=4):
    """What a user assembles today: a fresh eval-mode model, predict + ce_loss + MetricAccumulator per batch."""
    from uaps_b200.losses import ce_loss
    from uaps_b200.metrics import MetricAccumulator
    m = _small_model(C=C).eval()
    m.load_state_dict(model_state)
    acc = MetricAccumulator(DEV)
    ces = []
    for x, y in zip(xs, ys):
        logits = m.predict(x)
        ces.append(ce_loss(logits, y).item())
        acc.update(logits, y)
    r = acc.result()
    r["ce"] = sum(ces) / len(ces)
    return r


def test_validator_between_training_epochs():
    from uaps_b200.train import UAPSConfig, UAPSTrainer
    from uaps_b200.validate import Validator
    model = _small_model().train()
    val = Validator(model)                                   # before the trainer re-homes the parameters: must not matter
    trainer = UAPSTrainer(model, UAPSConfig(graph_warmup=1))
    g = torch.Generator(device=DEV).manual_seed(3)
    xl, xu = torch.randn(2, 3, 64, 64, generator=g, device=DEV), torch.randn(2, 3, 64, 64, generator=g, device=DEV)
    yl = ((xl[:, 0] > 0).long() + 2 * (xl[:, 1] > 0.5).long())
    xs, ys = _val_data(4)
    results = []
    for epoch in range(2):
        for _ in range(3):
            trainer.step(xl, yl, xu)
        assert model.training
        val.begin()
        for x, y in zip(xs, ys):
            val.update(x, y)
        res = val.result()
        ref = _reference_epoch(model.state_dict(), xs, ys)
        for k in ("pixel_accuracy", "mIoU", "mDice"):
            assert res[k] == pytest.approx(ref[k], rel=1e-12, abs=1e-15), (epoch, k)
        assert res["ce"] == pytest.approx(ref["ce"], rel=1e-6)
        assert res["val_loss"] == pytest.approx(ref["ce"] + 1 - ref["mDice"], rel=1e-6)
        assert res["batches"] == 4 and val.captures == 1    # one capture for the whole run
        results.append(res)
    assert results[0]["ce"] != results[1]["ce"]             # the second epoch saw the new weights
    assert len(trainer._graphs) == 1


def test_predict_is_unchanged_by_a_validator_and_the_mode_is_kept():
    from uaps_b200.validate import Validator
    m = _small_model().eval()
    xs, ys = _val_data(2)
    before = m.predict(xs[0]).clone()
    val = Validator(m)
    val.begin()
    for x, y in zip(xs, ys):
        val.update(x, y)
        val.update(x, y)
    val.result()
    assert not m.training and torch.equal(m.predict(xs[0]), before)


def test_fp32_path_uses_predict_in_eval_mode_and_restores_the_mode():
    from uaps_b200.validate import Validator
    m = _small_model(compute="fp32").train()
    xs, ys = _val_data(3)
    val = Validator(m)
    val.begin()
    for x, y in zip(xs, ys):
        val.update(x, y)
    res = val.result()
    assert m.training and val.captures == 0
    m.eval()
    from uaps_b200.losses import ce_loss
    from uaps_b200.metrics import MetricAccumulator
    acc, ces = MetricAccumulator(DEV), []
    for x, y in zip(xs, ys):
        logits = m.predict(x)
        ces.append(ce_loss(logits, y).item())
        acc.update(logits, y)
    ref = acc.result()
    assert res["mDice"] == pytest.approx(ref["mDice"], rel=1e-12) and res["ce"] == pytest.approx(sum(ces) / 3, rel=1e-6)


# ---- two processes, each holding half of every batch (needs two GPUs) -------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from uaps_b200.unet import UNet_UAPS
        from uaps_b200.validate import Validator
        torch.manual_seed(0)
        m = UNet_UAPS(3, 4).to(dev)
        g = torch.Generator().manual_seed(1)
        xs = [torch.randn(4, 3, 64, 64, generator=g) for _ in range(3)]
        per = 4 // world
        val = Validator(m)
        val.begin()
        for x in xs:
            y = ((x[:, 0] > 0).long() + 2 * (x[:, 1] > 0.5).long())
            val.update(x[rank * per:(rank + 1) * per].to(dev), y[rank * per:(rank + 1) * per].to(dev))
        q.put((rank, val.result()))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_give_the_full_batch_result():
    import torch.multiprocessing as mp
    from uaps_b200.validate import Validator
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=600) for _ in procs)
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    torch.manual_seed(0)
    from uaps_b200.unet import UNet_UAPS
    m = UNet_UAPS(3, 4).to(DEV)
    g = torch.Generator().manual_seed(1)
    xs = [torch.randn(4, 3, 64, 64, generator=g) for _ in range(3)]
    val = Validator(m)
    val.begin()
    for x in xs:
        val.update(x.to(DEV), ((x[:, 0] > 0).long() + 2 * (x[:, 1] > 0.5).long()).to(DEV))
    want = val.result()
    for r in (0, 1):
        for k in ("val_loss", "ce", "pixel_accuracy", "mIoU", "mDice"):
            assert got[r][k] == pytest.approx(want[k], rel=1e-9), (r, k)
        assert got[r]["batches"] == 3
