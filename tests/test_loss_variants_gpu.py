"""GPU parity of every fused-loss kernel variant, against the oracle run on the same device.

For each K in 1..6 and C in 2..8 the launcher (fused_loss.cu: pick_vec / pick_impl, fused_loss_impl.cuh: launch_kc)
instantiates three widths of pass 1 and pass 2, each supervised, unlabeled, and unlabeled with device-resident mix
weights (WDEV):

    |        | 4 px / thread                                  | 2 px / thread                                  | scalar                                     |
    | pass 1 | K*C <= 16, HW % 4 == 0, 16-B aligned planes    | K*C <= 24 and a 2-wide layout (or K*C in 17..24) | K*C > 24, odd HW, 4-B alignment, EXACT |
    | pass 2 | K*C <= 12 (same layout)                        | 13 <= K*C <= 24, or a 2-wide layout            | as above                                   |

A 2-wide layout is HW % 4 == 2 or planes that are only 8-byte aligned.  `_widths` restates that table and every
assertion message names the pair of kernels the case ran.  The ABI only asks for 4-byte aligned planes, so
contiguous views that start 1 or 2 floats into a larger buffer are legal inputs and reach the narrower kernels.

References: ``unlabeled_loss_ref`` / ``supervised_loss_ref`` as torch CUDA ops (bit-exact comparator for the
pseudo-label) and, for unlabeled gradients, ``unlabeled_loss_fp64_closed_form``.  Tolerances as in test_loss_gpu.py:
pseudo-label exact; scalars 1e-5 relative (default arithmetic: + 3e-8 absolute on l_uncert, 3e-9 on loss_u);
exp-var maps and gradients 1e-5 of the tensor's max; gradients against the fp64 closed form 2e-5.

K = 1: the mean prediction is the one softmax, so every KL map is 0 in exact arithmetic.  The oracle's map is
log(softmax) - log_softmax, i.e. rounding noise: per pixel |V| <= sum_c q_c |err_c| with |err_c| a few ulp of
|log q_c| + 1, which with sum_c q_c |log q_c| <= ln 8 stays below ~1.5e-6.  The kernel's map is a different noise of
the same size (exactly 0 in the default arithmetic).  l_uncert therefore gets an absolute floor of 2e-6 at K = 1
(and loss_u cw2 times that); a relative bound on a mean of noise says nothing.  K identical decoders are the same
case and get the same floor.

Large margins (a class M nats below its decoder's max): ex2.approx.ftz flushes p to 0 beyond ~87.3 nats, IEEE expf
beyond ~104; subnormal p and q appear in between.  The kernels must stay finite everywhere, match the oracle's
forward (finite everywhere here), match the fp64 closed form's gradients, and match torch's autograd where that is
finite (q_c > 0, i.e. M < 104 or the class is deep in only some decoders).
"""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle.uaps_loss_ref import (dice_loss_ref, supervised_loss_ref, unlabeled_loss_fp64_closed_form,
                                  unlabeled_loss_ref)

pytestmark = pytest.mark.gpu
REL = 1e-5
CW1, CW2 = 0.3, 0.2
K1_UNCERT_FLOOR = 2e-6             # see the module docstring


def _dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def _assert_close(a, b, what, rel=REL):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    assert torch.isfinite(a).all(), f"{what}: non-finite values"
    scale = b.abs().max().item() + 1e-30
    err = (a - b).abs().max().item()
    assert err <= rel * scale, f"{what}: max err {err:.3e} vs scale {scale:.3e}"


def _widths(K, C, avail, exact=False):
    """(pass-1, pass-2) pixels per thread the launcher picks for `avail` = the widest width the layout allows."""
    if exact:
        return 1, 1
    p1 = 4 if (avail == 4 and K * C <= 16) else (2 if (avail >= 2 and K * C <= 24) else 1)
    p2 = 4 if (avail == 4 and K * C <= 12) else (2 if (avail >= 2 and K * C <= 24) else 1)
    return p1, p2


def _mix(K, seed=1337):
    return np.random.default_rng(seed + K).dirichlet(np.ones(K))


def _place(tensors, offsets):
    """Each [B,C,H,W] tensor copied into a fresh buffer starting `off` floats in: a contiguous view whose data
    pointer is only 4 * off-byte aligned (torch's allocations are 512-byte aligned)."""
    out = []
    for t, off in zip(tensors, offsets):
        buf = torch.zeros(t.numel() + off + 4, device=t.device)
        v = buf[off:off + t.numel()].view(t.shape)
        v.copy_(t)
        assert v.data_ptr() % 16 == (4 * off) % 16
        out.append(v)
    return out


def _randn(K, C, B, H, W, seed, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(B, C, H, W, generator=g) * scale).to(_dev()) for _ in range(K)]


def check_unlabeled(z, mix_w, exact, what, autograd=True, cw1=CW1, cw2=CW2):
    """Fused unlabeled loss vs the oracle (forward, autograd) and the fp64 closed form; returns our outputs."""
    from uaps_b200.losses import uaps_unlabeled_loss
    K = len(z)
    zr = [t.detach().clone().requires_grad_(True) for t in z]
    ref = unlabeled_loss_ref(zr, mix_w, cw1, cw2)
    zs = [t.detach().requires_grad_(True) for t in z]          # no clone: keep the caller's alignment
    loss, ps, unc, pseudo, ev = uaps_unlabeled_loss(zs, mix_w, cw1, cw2, return_pseudo=True, return_exp_var=True,
                                                    exact_math=exact)
    grads = torch.autograd.grad(loss, zs)
    assert torch.equal(pseudo, ref["pseudo"]), \
        f"{what}: {(pseudo != ref['pseudo']).sum().item()} pseudo-labels of {pseudo.numel()} differ"
    noise = K == 1 or all(torch.equal(t, z[0]) for t in z)        # q is each decoder's softmax: V is rounding noise
    fl = K1_UNCERT_FLOOR if noise else (0.0 if exact else 3e-8)
    floor = {"loss_u": cw2 * fl if noise else (0.0 if exact else 3e-9), "ps_loss": 0.0, "l_uncert": fl}
    for key, v in (("loss_u", loss), ("ps_loss", ps), ("l_uncert", unc)):
        assert np.isfinite(v.item()), (what, key)
        assert v.item() == pytest.approx(ref[key].item(), rel=REL, abs=floor[key]), (what, key)
    _assert_close(torch.stack(ev), torch.stack(ref["exp_var"]).detach(), f"{what} exp_var")
    g = torch.stack(grads)
    cf = unlabeled_loss_fp64_closed_form(z, mix_w, cw1, cw2, ref["pseudo"])
    _assert_close(g, torch.stack(cf["dz"]), f"{what} grads vs fp64 closed form", rel=2e-5)
    if autograd:
        gr = torch.stack(torch.autograd.grad(ref["loss_u"], zr))
        assert torch.isfinite(gr).all(), f"{what}: the oracle's autograd was expected to be finite here"
        _assert_close(g, gr, f"{what} grads vs autograd")
    return dict(loss_u=loss, ps_loss=ps, l_uncert=unc, pseudo=pseudo, exp_var=ev, grads=grads)


def check_supervised(z, labels, exact, what):
    """Fused supervised loss vs the oracle; the upstream gradient reaches all three differentiable outputs."""
    from uaps_b200.losses import uaps_supervised_loss
    zr = [t.detach().clone().requires_grad_(True) for t in z]
    ref = supervised_loss_ref(zr, labels)
    gr = torch.autograd.grad(ref["supervised_loss"] + 0.3 * ref["total_loss_ce"] + 0.7 * ref["total_loss_dice"], zr)
    zs = [t.detach().requires_grad_(True) for t in z]
    sup, tce, tdice, ce_k = uaps_supervised_loss(zs, labels, exact_math=exact)
    g = torch.autograd.grad(sup + 0.3 * tce + 0.7 * tdice, zs)
    for key, v in (("supervised_loss", sup), ("total_loss_ce", tce), ("total_loss_dice", tdice)):
        assert np.isfinite(v.item()), (what, key)
        assert v.item() == pytest.approx(ref[key].item(), rel=REL), (what, key)
    np.testing.assert_allclose(ce_k.cpu().numpy(), torch.stack(ref["ce"]).detach().cpu().numpy(), rtol=REL,
                               err_msg=what)
    _assert_close(torch.stack(g), torch.stack(gr), f"{what} grads vs autograd")


# ---- A. the variant matrix ---------------------------------------------------------------------------------------
# layout -> (B, H, W, per-decoder float offsets, widest width it allows)
LAYOUTS = {
    "hw%4=0": ((2, 32, 36), (0,), 4),
    "hw%4=2": ((2, 30, 35), (0,), 2),
    "odd-hw": ((2, 31, 33), (0,), 1),
    "8B-aligned": ((2, 32, 36), (2,), 2),
    "4B-aligned": ((2, 32, 36), (1,), 1),
}


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("sup", [False, True], ids=["unlabeled", "supervised"])
@pytest.mark.parametrize("C", range(2, 9))
@pytest.mark.parametrize("K", range(1, 7))
def test_variant_matrix(K, C, sup, layout):
    (B, H, W), offs, avail = LAYOUTS[layout]
    z = _place(_randn(K, C, B, H, W, 100 * K + C), offs * K)
    what = f"K={K} C={C} {layout}: pass1/pass2 {_widths(K, C, avail)} px/thread"
    if sup:
        labels = torch.randint(0, C, (B, H, W), generator=torch.Generator().manual_seed(C)).to(_dev())
        check_supervised(z, labels, False, what)
    else:
        check_unlabeled(z, _mix(K), False, what)


@pytest.mark.parametrize("sup", [False, True], ids=["unlabeled", "supervised"])
@pytest.mark.parametrize("C", range(2, 9))
@pytest.mark.parametrize("K", range(1, 7))
def test_variant_matrix_exact(K, C, sup):
    """UAPS_LOSS_EXACT: the torch-order scalar kernels, whatever the layout."""
    z = _randn(K, C, 2, 30, 35, 200 * K + C)
    what = f"K={K} C={C} exact"
    if sup:
        labels = torch.randint(0, C, (2, 30, 35), generator=torch.Generator().manual_seed(C)).to(_dev())
        check_supervised(z, labels, True, what)
    else:
        check_unlabeled(z, _mix(K), True, what)


@pytest.mark.parametrize("K,C,offs", [(4, 4, (0, 2, 0, 2)), (3, 5, (2, 0, 1)), (2, 2, (0, 2))])
def test_planes_with_different_alignments(K, C, offs):
    """The width is the narrowest any decoder's planes allow: (0, 2, ...) floats in -> 2 px/thread, a 1 -> scalar."""
    z = _place(_randn(K, C, 2, 32, 36, 7 * K + C), offs)
    avail = 1 if 1 in offs else 2
    labels = torch.randint(0, C, (2, 32, 36), generator=torch.Generator().manual_seed(5)).to(_dev())
    what = f"K={K} C={C} offsets {offs}: {_widths(K, C, avail)} px/thread"
    check_unlabeled(z, _mix(K), False, what)
    check_supervised(z, labels, False, what)


# ---- B. large-margin logits ----------------------------------------------------------------------------------------
def _deep_logits(K, C, M, every, seed, same=False):
    """Background N(0, 2^2) logits [1, C, 16, 24].  At every third pixel half of the classes sit M nats below the
    max of the rest (random values); at the pixels after those, every class is 0 except class C - 1 at -M (the
    softmax's sum is then C - 1, which gives subnormal p and q between ~85.4 and ~87.3 nats).  `every`: in every
    decoder, so q_c underflows with p_kc; otherwise only in the first half of the decoders (q_c > 0).  `same`: all
    decoders identical (V ~ 0)."""
    g = torch.Generator().manual_seed(seed)
    B, H, W = 1, 16, 24
    idx = torch.arange(B * H * W).view(B, 1, H, W)
    cls = torch.arange(C).view(1, C, 1, 1)
    deep_a = (idx % 3 == 0) & (cls % 2 == idx % 2)          # half of the classes, alternating by pixel
    deep_b = (idx % 3 == 1).expand(B, C, H, W)
    flat = torch.where(cls == C - 1, -float(M), 0.0).expand(B, C, H, W)
    out = []
    for k in range(K):
        z = torch.randn(B, C, H, W, generator=g) * 2
        if every or k < (K + 1) // 2:
            top = z.masked_fill(deep_a, -float("inf")).amax(1, keepdim=True)
            z = torch.where(deep_a, top - M, z)
            z = torch.where(deep_b, flat, z)
        out.append(z)
    if same:
        out = [out[0].clone() for _ in range(K)]
    return [t.to(_dev()) for t in out]


MARGINS = [40.0, 80.0, 86.5, 90.0, 100.0, 120.0, 300.0]


@pytest.mark.parametrize("every", [True, False], ids=["all-decoders", "some-decoders"])
@pytest.mark.parametrize("M", MARGINS)
@pytest.mark.parametrize("C", [2, 4, 8])
@pytest.mark.parametrize("K", [1, 2, 4, 6])
def test_large_margins(K, C, M, every):
    if K == 1 and not every:
        pytest.skip("one decoder: 'some decoders' is all of them")
    z = _deep_logits(K, C, M, every, seed=31 * K + C)
    labels = torch.randint(0, C, (1, 16, 24), generator=torch.Generator().manual_seed(K)).to(_dev())
    torch_finite = M < 103.0 or not every          # fp32 q_c > 0, so torch's d xlogy(q, q)/dq is finite
    for exact in (False, True):
        what = f"K={K} C={C} M={M} {'all' if every else 'some'} {'exact' if exact else 'default'}"
        check_unlabeled(z, _mix(K), exact, what, autograd=torch_finite)
        check_supervised(z, labels, exact, what)        # labels fall on deep classes too: CE up to M per pixel


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_large_margins_identical_decoders(exact):
    """All decoders equal: V ~ 0 and E ~ 1 at every pixel, including those whose deep classes underflow."""
    for M in (90.0, 300.0):
        z = _deep_logits(4, 4, M, True, seed=5, same=True)
        o = check_unlabeled(z, _mix(4), exact, f"identical M={M}", autograd=M < 103.0)
        assert torch.stack(o["exp_var"]).min().item() > 0.999


@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
def test_decoders_disagree_strongly(exact):
    """Decoder k puts class k % C 300 nats above the others: V_k ~ 150-225 nats, so E_k underflows to 0."""
    K, C = 4, 4
    z = _randn(K, C, 1, 16, 24, 77)
    for k in range(K):
        z[k][:, k % C] += 300.0
    o = check_unlabeled(z, _mix(K), exact, "disagreeing decoders")
    assert torch.stack(o["exp_var"]).max().item() == 0.0
    labels = torch.randint(0, C, (1, 16, 24), generator=torch.Generator().manual_seed(2)).to(_dev())
    check_supervised(z, labels, exact, "disagreeing decoders")


@pytest.mark.parametrize("M", [86.5, 90.0, 120.0, 300.0])
def test_ensemble_head_large_margins(M):
    """ensemble_head.cu reuses the loss's per-pixel forward (pixel_mean_forward -> kl_terms): finite uncertainty equal
    to the oracle's when classes underflow in every decoder."""
    from uaps_b200.ensemble import ensemble_uncertainty
    for K, C in ((4, 8), (3, 4), (2, 2)):
        z = _deep_logits(K, C, M, True, seed=11 * K + C)
        ref = unlabeled_loss_ref(z, [1.0 / K] * K, 0.0, 0.0)
        acc = ref["soft"][0]
        vsum = ref["var"][0]
        for k in range(1, K):
            acc, vsum = acc + ref["soft"][k], vsum + ref["var"][k]
        q, unc = acc / K, vsum / K
        out = ensemble_uncertainty(z, return_probs=True)
        assert torch.isfinite(out.uncertainty).all() and torch.isfinite(out.image_uncertainty).all(), (K, C, M)
        assert torch.equal(out.labels.long(), torch.argmax(q, 1)), (K, C, M)
        assert (out.uncertainty - unc).abs().max().item() <= 1e-5 * max(unc.abs().max().item(), 0.1), (K, C, M)
        assert (out.mean_prob - q).abs().max().item() <= 1e-5 * q.abs().max().item(), (K, C, M)


# ---- C. supervised edges -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
@pytest.mark.parametrize("C", [2, 8])
def test_supervised_edges(C, exact):
    K, B, H, W = 4, 2, 24, 32
    z = _randn(K, C, B, H, W, 40 + C)
    g = torch.Generator().manual_seed(C)
    labels = torch.randint(0, C, (B, H, W), generator=g).to(_dev())
    # the label class 100 nats below the max at every 7th pixel: per-pixel CE ~ 100
    tail = (torch.arange(B * H * W, device=_dev()).view(B, H, W) % 7 == 0)
    for k in range(K):
        zl = z[k].gather(1, labels.unsqueeze(1))
        others = z[k].scatter(1, labels.unsqueeze(1), -1e30).amax(1, keepdim=True)
        z[k].scatter_(1, labels.unsqueeze(1), torch.where(tail.unsqueeze(1), others - 100.0, zl))
    check_supervised(z, labels, exact, f"C={C} label in the tail")
    # one class absent from the whole batch: its Dice term is 2*0/(card + eps) (card = sum of its probabilities)
    absent = labels.clamp(max=C - 2)
    check_supervised(z, absent, exact, f"C={C} class {C - 1} absent")
    # a single-class batch: every other class's Dice term is 0/(card + eps)
    check_supervised(z, torch.zeros_like(labels), exact, f"C={C} single class")
    check_supervised(z, torch.full_like(labels, C - 1), exact, f"C={C} single class {C - 1}")


# ---- D. sizes ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 2), (1, 1, 3), (1, 1, 5), (1, 1, 127), (1, 1, 129), (1, 17, 241),
                                   (3, 1, 1), (2, 1, 2), (1, 1, 4), (3, 2, 6)])
@pytest.mark.parametrize("K,C", [(4, 4), (2, 3), (6, 8)])
def test_tiny_and_ragged_sizes(K, C, shape):
    """Most threads idle and most blocks fold zero partials."""
    B, H, W = shape
    z = _randn(K, C, B, H, W, 9 * K + C + H * W)
    labels = torch.randint(0, C, (B, H, W), generator=torch.Generator().manual_seed(H * W)).to(_dev())
    for exact in (False, True):
        what = f"K={K} C={C} {shape} {'exact' if exact else 'default'}"
        check_unlabeled(z, _mix(K), exact, what)
        check_supervised(z, labels, exact, what)


def test_grid_stride_wraps():
    """2 x 512 x 512 px at K = C = 4: more pixel groups than the capped grid (<= 640 blocks x 128 threads) holds, so
    every thread's grid-stride loop runs several times in both passes."""
    K, C, B, H, W = 4, 4, 2, 512, 512
    assert B * H * W // 4 > 640 * 128
    g = torch.Generator(device=_dev()).manual_seed(3)
    z = [torch.randn(B, C, H, W, generator=g, device=_dev()) * 2 for _ in range(K)]
    check_unlabeled(z, _mix(K), False, "2x512x512")
    labels = torch.randint(0, C, (B, H, W), generator=g, device=_dev())
    check_supervised(z, labels, False, "2x512x512")


# ---- E. device-resident weights -------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(2, 32, 36), (2, 31, 33)])
@pytest.mark.parametrize("K,C", [(2, 4), (4, 4), (5, 2)])
def test_device_step_state_is_bitwise_the_by_value_call(K, C, shape):
    from uaps_b200.losses import uaps_supervised_loss, uaps_unlabeled_loss
    from uaps_b200.stepctx import DeviceStepState
    dev = _dev()
    z = _randn(K, C, *shape, 50 + K)
    mix_w = _mix(K)
    ds = DeviceStepState(dev, 1e-3)
    ds._view("mix_w")[:K] = torch.tensor(np.asarray(mix_w, np.float32), device=dev)
    ds.set("cw1", CW1)
    ds.set("cw2", CW2)

    def run(step_state):
        zs = [t.clone().requires_grad_(True) for t in z]
        out = uaps_unlabeled_loss(zs, mix_w if step_state is None else None, CW1, CW2, return_pseudo=True, return_exp_var=True,
                                  step_state=step_state)
        return out, torch.autograd.grad(out[0], zs)

    (a, ga), (b, gb) = run(None), run(ds)
    for x, y in zip(a[:4], b[:4]):
        assert torch.equal(x, y)
    assert all(torch.equal(x, y) for x, y in zip(a[4], b[4]))
    assert all(torch.equal(x, y) for x, y in zip(ga, gb))
    labels = torch.randint(0, C, (shape[0], shape[1], shape[2]), generator=torch.Generator().manual_seed(1)).to(dev)
    outs = []
    for step_state in (None, ds):
        zs = [t.clone().requires_grad_(True) for t in z]
        s = uaps_supervised_loss(zs, labels, step_state=step_state)
        outs.append((s, torch.autograd.grad(s[0], zs)))
    assert all(torch.equal(x, y) for x, y in zip(outs[0][0], outs[1][0]))
    assert all(torch.equal(x, y) for x, y in zip(outs[0][1], outs[1][1]))


# ---- F. pass 1 + finalize (the fallback when no peer-memory exchange exists) -----------------------------------------
def _pass1(L, lib, z, mix, labels, want_maps):
    K, (B, C, H, W) = len(z), z[0].shape
    dev = z[0].device
    ws = torch.zeros(lib.uaps_loss_workspace_bytes(K, C), dtype=torch.uint8, device=dev)
    sums = torch.empty(lib.uaps_loss_sums_count(K, C), dtype=torch.float64, device=dev)
    pseudo = torch.empty(B, H, W, dtype=torch.int64, device=dev) if want_maps else None
    ev = [torch.empty(B, H, W, device=dev) for _ in range(K)] if want_maps else None
    L.check(lib.uaps_loss_pass1(L.ptr_array(z), K, B, C, H * W, None if labels is not None else L.float_array(mix),
                                None if labels is None else labels.data_ptr(), ws.data_ptr(), sums.data_ptr(),
                                None if pseudo is None else pseudo.data_ptr(), None if ev is None else L.ptr_array(ev),
                                0, L.stream_ptr()), "uaps_loss_pass1")
    return sums, pseudo, ev


def _finalize(L, lib, sums, K, C, N, sup):
    sc = torch.empty(lib.uaps_loss_scalars_count(K, C), dtype=torch.float32, device=sums.device)
    L.check(lib.uaps_loss_finalize(sums.data_ptr(), K, C, N, CW1, CW2, int(sup), sc.data_ptr(), L.stream_ptr()),
            "uaps_loss_finalize")
    return sc


def _pass2(L, lib, z, mix, labels, sc, grad_out):
    K, (B, C, H, W) = len(z), z[0].shape
    dz = [torch.empty_like(t) for t in z]
    L.check(lib.uaps_loss_pass2(L.ptr_array(z), K, B, C, H * W, None if labels is not None else L.float_array(mix),
                                None if labels is None else labels.data_ptr(), sc.data_ptr(), grad_out.data_ptr(),
                                L.ptr_array(dz), 0, None, L.stream_ptr()), "uaps_loss_pass2")
    return torch.stack(dz)


@pytest.mark.parametrize("sup", [0, 1])
def test_pass1_finalize_and_sharding(sup):
    from uaps_b200 import _lib as L
    lib = L.lib()
    dev = _dev()
    K, C, B, H, W = 4, 4, 4, 64, 64           # a half batch is 2048 pixel groups = 16 whole blocks of pass 1
    z = _randn(K, C, B, H, W, 61)
    mix = _mix(K)
    labels = torch.randint(0, C, (B, H, W), generator=torch.Generator().manual_seed(4)).to(dev) if sup else None
    N = B * H * W
    # the same batch through pass1 + finalize and through pass1_scalars
    sums, pseudo, ev = _pass1(L, lib, z, mix, labels, not sup)
    sc = _finalize(L, lib, sums, K, C, N, sup)
    ws = torch.zeros(lib.uaps_loss_workspace_bytes(K, C), dtype=torch.uint8, device=dev)
    sums1 = torch.empty_like(sums)
    sc1 = torch.empty_like(sc)
    L.check(lib.uaps_loss_pass1_scalars(L.ptr_array(z), K, B, C, H * W, None if sup else L.float_array(mix),
                                        None if labels is None else labels.data_ptr(), ws.data_ptr(), sums1.data_ptr(),
                                        None, None, 0, CW1, CW2, sc1.data_ptr(), None, L.stream_ptr()), "pass1_scalars")
    torch.testing.assert_close(sums, sums1, rtol=1e-12, atol=0)
    torch.testing.assert_close(sc, sc1, rtol=1e-6, atol=0)
    # two half batches: pass 1 each, sums added in fp64, finalized with the global pixel count
    h = B // 2
    halves = [[t[:h].contiguous() for t in z], [t[h:].contiguous() for t in z]]
    lh = [None, None] if not sup else [labels[:h].contiguous(), labels[h:].contiguous()]
    parts = [_pass1(L, lib, halves[i], mix, lh[i], not sup) for i in range(2)]
    sums_sh = parts[0][0] + parts[1][0]
    torch.testing.assert_close(sums_sh, sums, rtol=1e-12, atol=0)
    sc_sh = _finalize(L, lib, sums_sh, K, C, N, sup)
    torch.testing.assert_close(sc_sh, sc, rtol=1e-6, atol=0)
    if not sup:
        assert torch.equal(torch.cat([parts[0][1], parts[1][1]]), pseudo)
        for k in range(K):
            assert torch.equal(torch.cat([parts[0][2][k], parts[1][2][k]]), ev[k])
    # pass 2 is per pixel given the scalars: each half's gradients are its slice of the full batch's, bit for bit
    grad_out = torch.zeros_like(sc)
    grad_out[L.SC_LOSS_U], grad_out[L.SC_PS_LOSS], grad_out[L.SC_L_UNCERT] = 1.0, 0.5, 0.25
    grad_out[L.SC_MEAN_CE], grad_out[L.SC_MEAN_DICE] = 0.3, 0.7
    full = _pass2(L, lib, z, mix, labels, sc_sh, grad_out)
    for i, sl in enumerate((slice(0, h), slice(h, B))):
        assert torch.equal(_pass2(L, lib, halves[i], mix, lh[i], sc_sh, grad_out), full[:, sl])
    assert torch.isfinite(full).all() and full.abs().max().item() > 0


# ---- G. per-decoder terms -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("exact", [False, True], ids=["default", "exact"])
@pytest.mark.parametrize("K,C", [(4, 4), (3, 2), (6, 7)])
def test_unlabeled_loss_terms(K, C, exact):
    from uaps_b200.losses import uaps_unlabeled_loss_terms
    z = _randn(K, C, 2, 32, 36, 90 + K * C)
    mix_w = _mix(K)
    ref = unlabeled_loss_ref(z, mix_w, CW1, CW2)
    loss, ps, unc, terms = uaps_unlabeled_loss_terms(z, mix_w, CW1, CW2, exact_math=exact)
    pseudo = ref["pseudo"]
    want = {"ps_k": torch.stack(ref["ps"]),
            "ebar_k": torch.stack([e.mean() for e in ref["exp_var"]]),
            "ce_k": torch.stack([F.cross_entropy(t, pseudo) for t in z]),
            "dice_k": torch.stack([dice_loss_ref(pseudo.unsqueeze(1), t) for t in z])}
    for key, w in want.items():
        assert terms[key].shape == (K,)
        np.testing.assert_allclose(terms[key].cpu().numpy(), w.detach().cpu().numpy(), rtol=REL, err_msg=key)
    assert loss.item() == pytest.approx(ref["loss_u"].item(), rel=REL, abs=0.0 if exact else 3e-9)
