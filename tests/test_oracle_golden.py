"""The oracle (oracle/iic_oracle.py, oracle/torch_port.py) against the reference's own outputs.

The golden vectors in tests/golden/ were produced by oracle/make_golden.py, which runs the
UNMODIFIED reference classes (fp64 and fp32).  These tests pin the restatement to them; they run
on CPU.  When the original project's source is provided (IIC_REFERENCE_ROOT, or the copy oracle/make_ref.py lays out
under oracle/_ref/) the reference is also re-run live.  The live tests use inputs of their own for which no reference
outputs are stored, so without the source they skip and what they check is not covered.
"""
import os
import sys

import numpy as np
import pytest

from conftest import golden_names, load_golden, relmax, ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_oracle as O  # noqa: E402
import ref_loader  # noqa: E402
import torch_port as TP  # noqa: E402

TOL = 1e-11  # fp64 restatement vs fp64 reference: only summation order differs


@pytest.mark.parametrize("name", golden_names("global"))
def test_global_oracle_matches_reference(name):
    g = load_golden(name)
    lamb = float(g["lamb"])
    loss, loss_nl, P = O.iid_loss(g["x"], g["y"], lamb)
    assert abs(loss - g["loss_f64"]) <= TOL * max(1, abs(g["loss_f64"]))
    assert abs(loss_nl - g["loss_no_lamb_f64"]) <= TOL * max(1, abs(g["loss_no_lamb_f64"]))
    assert relmax(P, g["P_f64"]) < TOL
    assert relmax(O.compute_joint(g["x"], g["y"], symmetric=False), g["joint_nosym_f64"]) < TOL
    gx, gy = O.iid_loss_grads(g["x"], g["y"], lamb)
    assert relmax(gx, g["gx_f64"]) < 1e-9 and relmax(gy, g["gy_f64"]) < 1e-9
    K = P.shape[0]
    w = np.linspace(-1.0, 1.0, K * K).reshape(K, K)
    fx, fy = O.iid_loss_grads(g["x"], g["y"], lamb, g_loss=0.7, g_loss_no_lamb=-0.3, g_P=w)
    assert relmax(fx, g["fullgx_f64"]) < 1e-9 and relmax(fy, g["fullgy_f64"]) < 1e-9


@pytest.mark.parametrize("name", golden_names("local"))
def test_local_oracle_matches_reference(name):
    g = load_golden(name)
    pad, lamda, patch = int(g["padding"]), float(g["lamda"]), int(g["patch_size"])
    mask = g.get("mask")
    if patch < 0:
        loss, gx, gy = O.iid_segmentation_loss(g["x"], g["y"], pad, lamda, mask, with_grads=True)
    else:
        loss, gx, gy = O.iid_segmentation_small_path_loss(g["x"], g["y"], pad, patch, lamda, mask,
                                                          with_grads=True)
    assert abs(loss - g["loss_f64"]) <= 1e-10 * max(1.0, abs(g["loss_f64"])), (loss, g["loss_f64"])
    assert relmax(gx, g["gx_f64"]) < 1e-8, relmax(gx, g["gx_f64"])
    assert relmax(gy, g["gy_f64"]) < 1e-8, relmax(gy, g["gy_f64"])


@pytest.mark.parametrize("name", golden_names("uda"))
def test_uda_oracle_matches_reference(name):
    g = load_golden(name)
    if str(g["kind"]) == "mse":
        loss, grad = O.mse_loss(g["prob"], g["target"], with_grads=True)
    else:
        loss, grad = O.kl_div(g["prob"], g["target"], weight=g.get("weight"), with_grads=True)
    assert abs(loss - g["loss_f64"]) <= 1e-12 * max(1.0, abs(g["loss_f64"]))
    assert relmax(grad, g["g_f64"]) < 1e-12


@pytest.mark.parametrize("name", golden_names("sup"))
def test_supervised_oracle_matches_reference(name):
    """semi_seg/epocher.py:165-166,183-184 as run by oracle/make_golden.py::run_sup."""
    g = load_golden(name)
    labels = g["labels"][:, 0]
    loss, grad = O.sup_kl_from_logits(g["logits"], labels, weight=g.get("weight"), with_grads=True)
    assert abs(loss - g["loss_f64"]) <= 1e-12 * max(1.0, abs(g["loss_f64"]))
    assert relmax(grad, g["g_f64"]) < 1e-11
    inter, union = O.dice_counts(g["logits"], labels)
    assert np.array_equal(inter, g["intersection"]) and np.array_equal(union, g["union"])
    dice = (2 * inter.sum(0) + 1e-6) / (union.sum(0) + 1e-6)
    assert relmax(dice, g["dice"]) < 1e-6          # the meter divides in float32


def test_supervised_oracle_rejects_bad_labels():
    with pytest.raises(AssertionError):
        O.class2one_hot(np.array([[[0, 4]]]), 4)


@pytest.mark.parametrize("name", golden_names("flip"))
def test_flip_oracle_matches_reference(name):
    """semi_seg/epocher.py:148-149,160-161,221-224 as run by oracle/make_golden.py::make_flip."""
    g = load_golden(name)
    flags = O.draw_flip_flags(int(g["seed"]), len(g["teacher"]))
    assert np.array_equal(flags, g["flags"])
    assert np.array_equal(O.flip_stack(g["teacher"], flags), g["teacher_tf"])
    loss, grad = O.uda_from_logits_flipped(g["student"], g["teacher"], flags, str(g["kind"]), with_grads=True)
    assert abs(loss - g["loss_f64"]) <= 1e-12 * max(1.0, abs(g["loss_f64"]))
    assert relmax(grad, g["g_f64"]) < 1e-11


def test_patch_windows_match_reference():
    g = load_golden("patch_windows")
    for key, wins in g.items():
        hw, ps = key.split("_p")
        h, w = (int(v) for v in hw.split("x"))
        ps = int(ps)
        got = O.patch_windows(h, w, (ps, ps), (ps // 2, ps // 2))
        assert [tuple(r) for r in wins.tolist()] == got, key


def test_simplex_matches_reference():
    g = load_golden("simplex_cases")
    for t, v in zip(g["cases"], g["verdicts"]):
        assert O.simplex(t) == bool(v)


def test_averaging_helpers():
    assert O.average_iter([1.0, 2.0, 6.0]) == 3.0
    assert abs(O.weighted_average_iter([1.0, 3.0], [0.25, 0.75]) - 2.5 / (1.0 + 1e-16)) < 1e-15


def test_softmax_roundtrip():
    rng = np.random.default_rng(0)
    z = rng.standard_normal((2, 5, 3, 4))
    p = O.softmax(z)
    assert O.simplex(p)
    g = rng.standard_normal(p.shape)
    num = np.zeros_like(z)
    eps = 1e-6
    for idx in np.ndindex(*z.shape):
        zp = z.copy(); zp[idx] += eps
        zm = z.copy(); zm[idx] -= eps
        num[idx] = ((O.softmax(zp) - O.softmax(zm)) * g).sum() / (2 * eps)
    assert relmax(O.softmax_backward(p, g), num) < 1e-6


# ---- the torch port (the timed CPU baseline) against the same goldens --------------------------
@pytest.mark.parametrize("name", golden_names("local"))
def test_torch_port_local(name):
    import torch
    g = load_golden(name)
    pad, lamda, patch = int(g["padding"]), float(g["lamda"]), int(g["patch_size"])
    x = torch.from_numpy(g["x"]).double().requires_grad_(True)
    y = torch.from_numpy(g["y"]).double().requires_grad_(True)
    m = None if "mask" not in g else torch.from_numpy(g["mask"]).double()
    if patch < 0:
        loss = TP.iid_segmentation_loss(x, y, pad, lamda, m)
    else:
        loss = TP.iid_segmentation_small_path_loss(x, y, pad, patch, lamda, m)
    gx, gy = torch.autograd.grad(loss, (x, y))
    assert abs(loss.item() - g["loss_f64"]) <= 1e-10 * max(1.0, abs(g["loss_f64"]))
    assert relmax(gx.numpy(), g["gx_f64"]) < 1e-8 and relmax(gy.numpy(), g["gy_f64"]) < 1e-8


@pytest.mark.parametrize("name", golden_names("global"))
def test_torch_port_global(name):
    import torch
    g = load_golden(name)
    x = torch.from_numpy(g["x"]).double().requires_grad_(True)
    y = torch.from_numpy(g["y"]).double().requires_grad_(True)
    loss, loss_nl, P = TP.iid_loss(x, y, float(g["lamb"]))
    assert abs(loss.item() - g["loss_f64"]) < 1e-11 * max(1, abs(g["loss_f64"]))
    assert abs(loss_nl.item() - g["loss_no_lamb_f64"]) < 1e-11 * max(1, abs(g["loss_no_lamb_f64"]))
    assert relmax(P.detach().numpy(), g["P_f64"]) < 1e-11


# ---- live re-run of the reference (when its source is provided) ---------------------------------
REF_MISSING = "the original project's source is not provided (IIC_REFERENCE_ROOT or oracle/_ref/reference)"


@pytest.mark.skipif(not ref_loader.available(), reason=REF_MISSING)
def test_live_reference_agrees_with_oracle_on_fresh_inputs():
    ns = ref_loader.load()
    torch = ns.torch
    rng = np.random.default_rng(7)
    x = torch.from_numpy(O.softmax(rng.standard_normal((2, 6, 13, 15)) * 2)).requires_grad_(True)
    y = torch.from_numpy(O.softmax(rng.standard_normal((2, 6, 13, 15)) * 2)).requires_grad_(True)
    loss = ns.IIDSegmentationSmallPathLoss(padding=2, patch_size=8)(x, y)
    gx, gy = torch.autograd.grad(loss, (x, y))
    l2, ox, oy = O.iid_segmentation_small_path_loss(x.detach().numpy(), y.detach().numpy(), 2, 8,
                                                    with_grads=True)
    assert abs(loss.item() - l2) < 1e-11
    assert relmax(ox, gx.numpy()) < 1e-8 and relmax(oy, gy.numpy()) < 1e-8


@pytest.mark.skipif(not ref_loader.available(), reason=REF_MISSING)
def test_live_reference_supervised_branch():
    ns = ref_loader.load()
    torch = ns.torch
    rng = np.random.default_rng(11)
    lg = torch.from_numpy(rng.standard_normal((2, 4, 10, 10)) * 2).requires_grad_(True)
    tgt = torch.from_numpy(rng.integers(0, 4, size=(2, 1, 10, 10)))
    loss = ns.KL_div(verbose=False)(lg.softmax(1), ns.class2one_hot(tgt.squeeze(1), 4))
    (g,) = torch.autograd.grad(loss, (lg,))
    ol, og = O.sup_kl_from_logits(lg.detach().numpy(), tgt.numpy()[:, 0], with_grads=True)
    assert abs(loss.item() - ol) < 1e-12 and relmax(og, g.numpy()) < 1e-11
    meter = ref_loader.load_dice()(C=4)
    meter.add(lg.detach().max(1)[1], tgt.squeeze(1))
    inter, union = O.dice_counts(lg.detach().numpy(), tgt.numpy()[:, 0])
    assert np.array_equal(meter._intersections[0].numpy(), inter)
    assert np.array_equal(meter._unions[0].numpy(), union)


@pytest.mark.skipif(not ref_loader.available(), reason=REF_MISSING)
def test_live_reference_flip_draws():
    ns = ref_loader.load()
    torch = ns.torch
    TensorRandomFlip, FixRandomSeed = ref_loader.load_flip()
    T = TensorRandomFlip(axis=[1, 2], threshold=0.8)
    x = torch.arange(9 * 2 * 3 * 5, dtype=torch.float32).reshape(9, 2, 3, 5)
    for seed in (0, 1, 7, 2**31 - 1):
        with FixRandomSeed(seed):
            ref = torch.stack([T(s) for s in x], dim=0)
        assert np.array_equal(O.flip_stack(x.numpy(), O.draw_flip_flags(seed, 9)), ref.numpy()), seed
