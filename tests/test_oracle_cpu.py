"""CPU suite: the oracle against the committed golden vectors (written by oracle/make_golden.py from the
imported reference), host-side logic, and the C-ABI library's exports.  No GPU, no /root/reference."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN, ROOT
from oracle.perturb_ref import dropout_ref, feature_dropout_ref, feature_noise_ref
from oracle.uaps_loss_ref import (consistency_weight_ref, sigmoid_rampup_ref, supervised_loss_ref,
                                  unlabeled_loss_fp64_closed_form, unlabeled_loss_ref)


def _run_case(c):
    z = [torch.from_numpy(a).clone().requires_grad_(True) for a in c["logits"]]
    out = unlabeled_loss_ref(z, c["mix_w"], float(c["cw"][0]), float(c["cw"][1]))
    out["loss_u"].backward()
    return z, out


def test_unlabeled_oracle_matches_golden(loss_cases):
    names = [n for n in loss_cases if not n.startswith("sup")]
    assert len(names) >= 9
    for name in names:
        c = loss_cases[name]
        z, out = _run_case(c)
        assert np.array_equal(out["pseudo"].numpy(), c["pseudo"]), name
        for key in ("loss_u", "ps_loss", "l_uncert"):
            assert out[key].item() == pytest.approx(float(c[key]), rel=1e-6), (name, key)
        np.testing.assert_allclose(torch.stack([e.detach() for e in out["exp_var"]]).numpy(), c["exp_var"],
                                   rtol=1e-6, atol=1e-7)
        g = torch.stack([t.grad for t in z]).numpy()
        np.testing.assert_allclose(g, c["grads"], rtol=1e-5, atol=1e-6 * np.abs(c["grads"]).max())


def test_closed_form_backward_matches_golden(loss_cases):
    for name, c in loss_cases.items():
        if name.startswith("sup"):
            continue
        z = [torch.from_numpy(a) for a in c["logits"]]
        cf = unlabeled_loss_fp64_closed_form(z, c["mix_w"], float(c["cw"][0]), float(c["cw"][1]),
                                             torch.from_numpy(c["pseudo"]))
        g = torch.stack(cf["dz"]).float().numpy()
        np.testing.assert_allclose(g, c["grads"], rtol=0, atol=2e-5 * np.abs(c["grads"]).max())
        assert cf["ps_loss"].item() == pytest.approx(float(c["ps_loss"]), rel=1e-5)
        assert cf["l_uncert"].item() == pytest.approx(float(c["l_uncert"]), rel=1e-5)


@pytest.mark.parametrize("every", [True, False])
@pytest.mark.parametrize("margin", [60.0, 95.0, 110.0, 300.0, 700.0])
def test_closed_form_matches_fp64_autograd_at_large_margins(margin, every):
    """The GPU loss tests take the fp64 closed form as the gradient reference where fp32 autograd of the oracle is NaN
    (a class more than ~104 nats below the max in every decoder: q_c = 0 and d xlogy(q, q)/dq = -inf).  In fp64, q_c
    stays positive up to ~745 nats, so autograd of the same oracle is finite there and the closed form must equal it."""
    K, C, B, H, W = 3, 4, 2, 4, 6
    g = torch.Generator().manual_seed(17)
    z = [torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 2 for _ in range(K)]
    pix = torch.arange(B * H * W).view(B, H, W) % 3 == 0
    for k in range(K if every else 1):                    # classes 2 and 3 `margin` nats below the max
        top = z[k][:, :2].amax(1)
        for c in (2, 3):
            z[k][:, c] = torch.where(pix, top - margin, z[k][:, c])
    mix_w = [0.5, 0.3, 0.2]
    zr = [t.clone().requires_grad_(True) for t in z]
    ref = unlabeled_loss_ref(zr, mix_w, 0.3, 0.2)
    ref["loss_u"].backward()
    auto = torch.stack([t.grad for t in zr])
    cf = unlabeled_loss_fp64_closed_form(z, mix_w, 0.3, 0.2, ref["pseudo"])
    dz = torch.stack(cf["dz"])
    assert torch.isfinite(auto).all() and torch.isfinite(dz).all()
    assert (dz - auto).abs().max().item() <= 1e-9 * auto.abs().max().item()
    assert cf["ps_loss"].item() == pytest.approx(ref["ps_loss"].item(), rel=1e-12)
    assert cf["l_uncert"].item() == pytest.approx(ref["l_uncert"].item(), rel=1e-12)


def test_ties_take_lowest_index(loss_cases):
    c = loss_cases["k4c4_ties"]
    # planes 1 == 0 and 3 == 2 in every decoder, so only labels 0 and 2 can win
    assert set(np.unique(c["pseudo"]).tolist()) <= {0, 2}


def test_supervised_oracle_matches_golden(loss_cases):
    c = loss_cases["sup_k4c4"]
    z = [torch.from_numpy(a).clone().requires_grad_(True) for a in c["logits"]]
    out = supervised_loss_ref(z, torch.from_numpy(c["labels"]))
    out["supervised_loss"].backward()
    assert out["supervised_loss"].item() == pytest.approx(float(c["supervised_loss"]), rel=1e-6)
    assert out["total_loss_ce"].item() == pytest.approx(float(c["total_loss_ce"]), rel=1e-6)
    assert out["total_loss_dice"].item() == pytest.approx(float(c["total_loss_dice"]), rel=1e-6)
    np.testing.assert_allclose(torch.stack([t.grad for t in z]).numpy(), c["grads"], rtol=1e-5, atol=1e-9)


def test_ramps_match_golden():
    from uaps_b200.ramps import get_current_consistency_weight, sigmoid_rampup
    g = np.load(os.path.join(GOLDEN, "ramps.npz"))
    for cur, val in zip(g["current"], g["sigmoid_rampup_200"]):
        assert sigmoid_rampup_ref(cur, 200.0) == pytest.approx(val, rel=1e-15)
        assert sigmoid_rampup(cur, 200.0) == pytest.approx(val, rel=1e-15)
    assert sigmoid_rampup(5, 0) == 1.0
    for it, w in zip(g["iters"], g["consistency_weight"]):
        assert consistency_weight_ref(int(it)) == pytest.approx(w, rel=1e-15)
        assert get_current_consistency_weight(int(it)) == pytest.approx(w, rel=1e-15)


def test_perturb_oracle_matches_golden():
    g = np.load(os.path.join(GOLDEN, "perturb.npz"))
    x = torch.from_numpy(g["x"])
    assert torch.equal(feature_noise_ref(x, torch.from_numpy(g["noise"])), torch.from_numpy(g["y_noise"]))
    assert torch.equal(dropout_ref(x, torch.from_numpy(g["keep"]), 0.5), torch.from_numpy(g["y_drop"]))
    assert torch.equal(feature_dropout_ref(x, float(g["u"])), torch.from_numpy(g["y_fd"]))


def test_unet_oracle_matches_golden():
    from oracle.unet_ref import feature_shapes, synthetic_rand, synthetic_state_dict, unet_uaps_ref
    g = np.load(os.path.join(GOLDEN, "unet_small.npz"))
    sd = synthetic_state_dict(3, 4)
    assert len(sd) == 334
    x = torch.from_numpy(g["x"])
    B, _, H, W = x.shape
    out = unet_uaps_ref(x, sd, synthetic_rand(feature_shapes(B, H, W)))
    ref = torch.from_numpy(g["out"])
    for k in range(4):
        assert (out[k] - ref[k]).abs().max().item() <= 1e-5 * ref[k].abs().max().item()


# ---- the C-ABI library: loads and exports exactly what include/uaps_b200.h declares ----------------
def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "uaps_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(uaps_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from uaps_b200 import _lib
    assert os.path.exists(_lib.LIB_PATH), "run `python -m uaps_b200.build` (or __graft_entry__.build()) first"
    handle = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 13
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/uaps_b200.h but not exported"
    assert sorted(_lib.exported_symbols()) == declared, "python binding and header diverge"
    lib = _lib.lib()
    assert lib.uaps_abi_version() == _lib.ABI_VERSION == 2
    # pure host-side queries (no GPU work)
    assert lib.uaps_loss_sums_count(4, 4) == 3 * 4 + 2 * 16 + 4
    assert lib.uaps_loss_scalars_count(4, 4) == 8 + 16 + 32
    assert lib.uaps_loss_sums_count(7, 4) == -2 and lib.uaps_loss_sums_count(4, 9) == -2
    assert lib.uaps_loss_workspace_bytes(4, 4) > 0
    assert b"range" in lib.uaps_error_string(-2)


def test_product_path_refuses_cpu_tensors():
    from uaps_b200.losses import uaps_unlabeled_loss
    z = [torch.randn(1, 4, 8, 8) for _ in range(4)]
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        uaps_unlabeled_loss(z, [0.25] * 4, 0.1, 0.1)


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "uaps_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


def test_metric_restatement_matches_reference_golden():
    """The loops of utilities/metrics.py:7-61 as restated for the GPU parity tests, against the outputs of the
    reference's own functions (tests/golden/metrics.npz, written by oracle/make_golden.py:golden_metrics)."""
    import numpy as np
    import torch
    import torch.nn.functional as F
    from conftest import load_cases
    for name, c in load_cases("metrics.npz").items():
        logits, m, C = torch.from_numpy(c["logits"]), torch.from_numpy(c["mask"]).view(-1), int(c["n_classes"])
        pred = torch.argmax(F.softmax(logits, dim=1), dim=1).view(-1)
        assert float(torch.eq(pred, m).sum()) / m.numel() == float(c["pixel_accuracy"]), name
        ious, dices = [], []
        for k in range(1, C):
            tc, tl = pred == k, m == k
            if tl.sum().item() == 0:
                ious.append(np.nan); dices.append(np.nan)
                continue
            inter, union = (tc & tl).sum().item(), (tc | tl).sum().item()
            ious.append((inter + 1e-10) / (union + 1e-10)); dices.append(2 * (inter + 1e-10) / (union + inter + 1e-10))
        assert np.nanmean(ious) == float(c["mIoU"]) and np.nanmean(dices) == float(c["mDice"]), name
