"""The training log on the GPU: the labeled batch's confusion counts written inside the iteration against
``metrics.confusion`` of the same logits, the scalars of captured replays against what each replay returned, no host sync
per iteration, an unchanged iteration with the log on, K = 5 and C = 2 shapes, and two ranks against the whole batch."""
import math
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _trainer(rows, C=4, cin=3, n_aux=3, seed=0, compute="bf16", **cfg):
    from uaps_b200.train import UAPSConfig, UAPSTrainer
    from uaps_b200.unet import UNet_UAPS
    torch.manual_seed(seed)
    model = UNet_UAPS(cin, C, n_aux=n_aux, compute=compute).to(DEV)
    return UAPSTrainer(model, UAPSConfig(num_classes=C, train_log_rows=rows, **cfg))


def _batches(n, B=4, H=64, W=64, C=4, cin=3, seed=4):
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(n):
        xl, xu = torch.randn(B, cin, H, W, generator=g).to(DEV), torch.randn(B, cin, H, W, generator=g).to(DEV)
        yl = ((xl[:, 0] > 0).long() + 2 * (xl[:, -1] > 0.5).long()) % C
        out.append((xl, yl, xu))
    return out


def _labeled_logits(model):
    """Forward hook: a clone of the model's first output on every call (the labeled forward is the first call of a step)."""
    seen = []
    handle = model.register_forward_hook(lambda m, inp, out: seen.append(out[0].detach().clone()))
    return seen, handle


def _row_scalars(out):
    from uaps_b200.train import LOG_SCALARS
    return torch.cat([torch.stack([out[k] for k in LOG_SCALARS]), out["loss_ce_k"]]).double()


@pytest.mark.parametrize("mode", ["device_eager", "host"])
def test_counts_are_exact(mode):
    """Every row's counts equal uaps_confusion of the labeled logits that iteration produced, and log_result's metrics
    are the per-row metrics_from_confusion averaged; the scalars are what step returned, bit for bit."""
    import numpy as np
    from uaps_b200.metrics import confusion, metrics_from_confusion
    C = 4
    tr = _trainer(8, cuda_graph=False)
    data = _batches(3)
    seen, handle = _labeled_logits(tr.model)
    tr.log_begin()
    outs = []
    for i, (xl, yl, xu) in enumerate(data):
        if mode == "host":
            out = tr.step(xl, yl, xu, mix_w=np.random.default_rng(i).dirichlet(np.ones(tr.k)))
        else:
            out = tr.step(xl, yl, xu)
        outs.append({k: v.clone() for k, v in out.items()})
    handle.remove()
    torch.cuda.synchronize()
    assert len(seen) == 2 * len(data)                        # labeled + unlabeled forward per step
    assert tr.log_state.tolist() == [3, 0, 0] and tr.log_counts[3:].abs().sum() == 0
    want = []
    for i, (xl, yl, _) in enumerate(data):
        conf = confusion(seen[2 * i], yl)
        row = tr.log_counts[i]
        assert torch.equal(row[:C * C].view(C, C).long(), conf), i
        assert row[C * C + 1].item() == row[C * C + 2].item() == yl.numel()
        assert torch.equal(tr.log_scalars[i], _row_scalars(outs[i])), i
        want.append([float(v) for v in metrics_from_confusion(conf, n_pixels=yl.numel())])
    res = tr.log_result()
    for j, k in enumerate(("pixel_accuracy", "mIoU", "mDice")):
        assert res[k] == pytest.approx(sum(w[j] for w in want) / len(want), rel=1e-12, abs=1e-15), k
    assert res["iterations"] == 3 and len(res["loss_ce_k"]) == tr.k


def test_captured_replays_add_one_row_each_with_the_returned_scalars():
    from uaps_b200.train import LOG_SCALARS
    tr = _trainer(16, graph_warmup=2)
    data = _batches(4)
    for i in range(3):                                       # two eager warm-up iterations, then capture + first replay
        tr.step(*data[i % 4])
    assert len(tr._graphs) == 1
    tr.log_begin()
    k, outs = 5, []
    for i in range(k):
        out = tr.step(*data[i % 4])
        outs.append({n: v.clone() for n, v in out.items()})
    torch.cuda.synchronize()
    assert len(tr._graphs) == 1 and tr.log_state.tolist() == [k, 0, 0]
    assert tr.log_scalars[k:].abs().sum() == 0 and tr.log_counts[k:].abs().sum() == 0
    rows = torch.stack([_row_scalars(o) for o in outs])
    assert torch.equal(tr.log_scalars[:k], rows)
    res = tr.log_result()
    mean = rows.mean(0).tolist()
    for j, n in enumerate(LOG_SCALARS):
        assert res[n] == pytest.approx(mean[j], rel=1e-12), n
    assert res["loss_ce_k"] == pytest.approx(mean[len(LOG_SCALARS):], rel=1e-12)
    assert res["iterations"] == k and 0.0 <= res["pixel_accuracy"] <= 1.0 and math.isfinite(res["mDice"])
    assert sum(tr.log_counts[i, :16].sum().item() for i in range(k)) == k * data[0][1].numel()


@pytest.mark.parametrize("graph", [True, False])
def test_no_host_sync_per_iteration(graph):
    """Captured: 5 replays.  Eager (cuda_graph=False): 2 iterations, where the log's Python (the head and
    uaps_val_scalars launches) runs every time -- the path the warm-up iterations take too."""
    tr = _trainer(16, graph_warmup=1, cuda_graph=graph)
    data = _batches(2)
    for i in range(2 if graph else 1):                       # warm-up (and capture)
        tr.step(*data[i])
    tr.log_begin()
    torch.cuda.synchronize()
    n = 5 if graph else 2
    torch.cuda.set_sync_debug_mode("error")
    try:
        for i in range(n):
            tr.step(*data[i % 2])
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert tr.log_result()["iterations"] == n and len(tr._graphs) == (1 if graph else 0)


# Run-to-run noise of the first iteration's scalars on the bf16 path, with or without the log: the BatchNorm statistics
# are summed with atomics (fp32 in shared memory, then fp64), so the logits vary at ~1e-7 relative and the scalars inherit
# it.  Measured on a B200, six log-off trainers in a fresh process: <= 1.7e-7 relative for loss / supervised_loss /
# total_loss_ce / total_loss_dice, 4.9e-7 for loss_ce_k, 5e-7 absolute (1e-5 relative) for l_uncert (a mean of differences
# of O(1) log terms), 4.8e-5 relative for ps_loss (one near-tie pixel of the 16 384 whose pseudo-label flips moves it by
# ~6e-5).  After the rest of the GPU suite had run in the same process, loss once differed by 1.5e-6 between two
# trainers.  The floors sit a few times above those figures; the spread of three log-off trainers is added on top.
_REL_FLOOR = {"loss": 5e-6, "supervised_loss": 5e-6, "total_loss_ce": 5e-6, "total_loss_dice": 5e-6, "loss_ce_k": 5e-6,
              "ps_loss": 3e-4, "l_uncert": 0.0}
_ABS_FLOOR = {"l_uncert": 3e-6}


def _first_step(rows, data, **kw):
    tr = _trainer(rows, **kw)
    before = tr.optimizer.flat_p.clone()
    out = tr.step(*data)
    return {k: v.clone() for k, v in out.items()}, tr.optimizer.flat_p - before


def _disagree(d, ref):
    """Share of the parameters Adam moved in ``ref`` that moved the other way (or not at all) in ``d``."""
    moved = ref != 0
    return (torch.sign(d) != torch.sign(ref))[moved].float().mean().item()


def test_the_iteration_is_unchanged_by_the_log():
    """bf16 path, same seed, weights and data: the log-on trainer's first iteration stays within the run-to-run noise of
    log-off trainers.  Scalars: a multiple of the spread of three log-off trainers plus the floors above.  Update: Adam's
    first step is +-lr where the gradient is not tiny, so the share of parameters moved the other way measures gradient
    noise (weight-gradient and BatchNorm atomics flip near-zero gradients; ~1 % of them on a B200): the log-on trainer
    may not disagree with the first log-off trainer much more than the other two do."""
    lr = 1e-3
    data = _batches(1)[0]
    offs = [_first_step(0, data) for _ in range(3)]
    on, d_on = _first_step(8, data)
    off, d_off = offs[0]
    for k in off:
        vals = torch.stack([o[k] for o, _ in offs])
        spread = vals.max(0).values - vals.min(0).values
        tol = 4 * spread + _REL_FLOOR[k] * off[k].abs() + _ABS_FLOOR.get(k, 0.0)
        diff = (on[k] - off[k]).abs()
        assert bool((diff <= tol).all()), (k, on[k].tolist(), vals.tolist())
    noise = max(_disagree(d, d_off) for _, d in offs[1:])
    assert _disagree(d_on, d_off) <= 2 * noise + 0.005, (_disagree(d_on, d_off), noise)
    assert (d_on - d_off).abs().max().item() <= 2.05 * lr


def test_the_reference_path_forward_is_bitwise_unchanged_by_the_log():
    """The fp32 reference path's forward with cuDNN in deterministic mode and injected draws (host mode) is reproducible,
    so there the log must not change the iteration's scalars at all: bit for bit, and the log's row holds the same bits.
    (Its backward still sums with atomics, so the update is left to the bf16 test above.)"""
    import numpy as np
    from uaps_b200 import perturb as P
    data = _batches(1)[0]
    mix_w = np.random.default_rng(3).dirichlet(np.ones(4))
    flags = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        res = {}
        for rows in (0, 8, 0):
            P.manual_seed(5)
            tr = _trainer(rows, compute="fp32")
            out = {k: v.clone() for k, v in tr.step(*data, mix_w=mix_w).items()}
            res.setdefault(rows, []).append(out)
            if rows:
                torch.cuda.synchronize()
                assert torch.equal(tr.log_scalars[0], _row_scalars(out)) and tr.log_result()["iterations"] == 1
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = flags
    (off, off2), (on,) = res[0], res[8]
    assert all(torch.equal(off[k], off2[k]) for k in off), "the fp32 forward is not reproducible"
    for k in off:
        assert torch.equal(on[k], off[k]), k


@pytest.mark.parametrize("cin,H,W,C,n_aux", [(3, 240, 640, 2, 4), (1, 512, 512, 2, 3)])
def test_k5_and_dagm_shapes(cin, H, W, C, n_aux):
    B = 2
    tr = _trainer(8, C=C, cin=cin, n_aux=n_aux, graph_warmup=1)
    data = _batches(2, B=B, H=H, W=W, C=C, cin=cin)
    tr.log_begin()
    losses = []
    for i in range(4):                                       # warm-up, capture + replay, two replays
        losses.append(tr.step(*data[i % 2])["loss"].clone())
    res = tr.log_result()
    assert len(tr._graphs) == 1 and res["iterations"] == 4
    assert len(res["loss_ce_k"]) == n_aux + 1 == tr.k and all(math.isfinite(v) for v in res["loss_ce_k"])
    assert res["loss"] == pytest.approx(torch.stack(losses).double().mean().item(), rel=1e-12)
    assert tr.log_counts.shape[1] == C * C + 3
    assert tr.log_counts[:4, :C * C].sum().item() == 4 * B * H * W
    assert 0.0 <= res["pixel_accuracy"] <= 1.0


# ---- two processes, each holding half of every labeled batch (needs two GPUs) -----------------------------------------
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
        from uaps_b200.train import UAPSConfig, UAPSTrainer
        from uaps_b200.unet import UNet_UAPS
        torch.manual_seed(0)
        tr = UAPSTrainer(UNet_UAPS(3, 4).to(dev), UAPSConfig(cuda_graph=False, train_log_rows=8))
        seen = []
        handle = tr.model.register_forward_hook(lambda m, inp, out: seen.append(out[0].detach().cpu()))
        g = torch.Generator().manual_seed(1)
        per = 4 // world
        tr.log_begin()
        for _ in range(3):
            xl, xu = torch.randn(4, 3, 64, 64, generator=g), torch.randn(4, 3, 64, 64, generator=g)
            yl = (xl[:, 0] > 0).long() + 2 * (xl[:, 1] > 0.5).long()
            sl = slice(rank * per, (rank + 1) * per)
            tr.step(xl[sl].to(dev), yl[sl].to(dev), xu[sl].to(dev))
        handle.remove()
        res = tr.log_result()
        q.put((rank, res, seen[0::2], tr.log_counts[:3].cpu()))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_count_the_whole_batch():
    import torch.multiprocessing as mp
    from uaps_b200.metrics import confusion, metrics_from_confusion
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = {r: rest for r, *rest in (q.get(timeout=600) for _ in procs)}
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    g = torch.Generator().manual_seed(1)
    want = []
    for i in range(3):
        xl, _ = torch.randn(4, 3, 64, 64, generator=g), torch.randn(4, 3, 64, 64, generator=g)
        yl = ((xl[:, 0] > 0).long() + 2 * (xl[:, 1] > 0.5).long()).to(DEV)
        logits = torch.cat([got[0][1][i], got[1][1][i]]).to(DEV)
        conf = confusion(logits, yl)
        summed = got[0][2][i] + got[1][2][i]
        assert torch.equal(summed[:16].view(4, 4).long(), conf.cpu()), i
        want.append([float(v) for v in metrics_from_confusion(conf, n_pixels=yl.numel())])
    for r in (0, 1):
        res = got[r][0]
        assert res["iterations"] == 3
        for j, k in enumerate(("pixel_accuracy", "mIoU", "mDice")):
            assert res[k] == pytest.approx(sum(w[j] for w in want) / 3, rel=1e-12, abs=1e-15), (r, k)
    assert got[0][0]["loss"] == pytest.approx(got[1][0]["loss"], rel=1e-6)
