"""The ignore label (``ignore_index``) of the fused supervised loss and its Dice counts, 1 to 256 classes.

The expected values come from the fp64 oracle applied to the pixels whose label is not the ignore label, gathered
into one (1, C, 1, n) map with (1, 1, n) labels: the loss is then the reference's ``KL_div`` mean over those n
pixels, and the gradient is scattered back with zeros at the ignored pixels.  The expected Dice counts are the
oracle's per sample, on that sample's kept pixels.  Bounds as everywhere in the suite: loss 1e-5 relative, gradient
1e-4 max-norm relative, Dice counts exact.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, relmax

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_oracle as O  # noqa: E402

LOSS_RTOL = 1e-5
GRAD_RTOL = 1e-4
NARROW_C = [2, 3, 4, 5, 8]
WIDE_C = [9, 16, 17, 19, 21, 32, 33, 64, 65, 128, 129, 150, 256]
# inner = 240 (% 4 == 0: 4 pixels per thread / lane, a partial last tile) and inner = 63 (% 4 != 0: 1 pixel)
SHAPES = [(2, 12, 20), (3, 7, 9)]
ONE_PIXEL = "one"                                # the ~0 % case: exactly one ignored pixel


@pytest.fixture(scope="module")
def iic(cuda_device):
    import iic_b200
    return iic_b200


def _logits(rng, shape, scale=2.0):
    return (rng.standard_normal(shape) * scale).astype(np.float32)


def _dev(a, dev, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t.requires_grad_(True) if grad else t


def _labels(rng, B, C, sp, ign, frac):
    """Labels in [0, C) with a fraction `frac` of the pixels (or exactly one for ONE_PIXEL) set to `ign`."""
    lab = rng.integers(0, C, size=(B,) + tuple(sp)).astype(np.int64)
    flat = lab.reshape(-1)
    if frac == ONE_PIXEL:
        flat[rng.integers(0, flat.size)] = ign
    else:
        flat[rng.random(flat.size) < frac] = ign
    return lab


def _expected(lg, lab, ign, weight=None):
    """(loss, d loss / d logits, intersection, union) of the oracle on the pixels whose label is not `ign`."""
    B, C = lg.shape[:2]
    z = lg.reshape(B, C, -1).astype(np.float64)
    lb = lab.reshape(B, -1)
    keep = lb != ign
    grad = np.zeros_like(z)
    if keep.any():
        cols = z.transpose(1, 0, 2)[:, keep]                              # (C, n)
        loss, g = O.sup_kl_from_logits(cols[None, :, None, :], lb[keep][None, None, :], weight=weight,
                                       with_grads=True)
        gz = grad.transpose(1, 0, 2)                                      # a view of grad
        gz[:, keep] = g[0, :, 0, :]
    else:
        loss = 0.0
    inter = np.zeros((B, C), np.int64)
    union = np.zeros((B, C), np.int64)
    for b in range(B):
        if keep[b].any():
            oi, ou = O.dice_counts(z[b][:, keep[b]][None, :, None, :], lb[b][keep[b]][None, None, :])
            inter[b], union[b] = oi[0], ou[0]
    return loss, grad.reshape(lg.shape), inter, union


def _run(iic, dev, lg, lab, ign, weight=None, scale=1.0):
    ld = _dev(lg, dev, grad=True)
    loss, (inter, union) = iic.sup_kl_from_logits(ld, _dev(lab, dev), weight=weight, return_dice=True,
                                                  ignore_index=ign)
    (scale * loss).backward()
    return loss.item(), ld.grad.cpu().numpy(), inter.cpu().numpy(), union.cpu().numpy()


def _check(got, want, scale=1.0):
    loss, grad, inter, union = got
    ol, og, oi, ou = want
    assert abs(loss - ol) <= LOSS_RTOL * abs(ol), (loss, ol)
    assert relmax(grad, scale * og) <= GRAD_RTOL
    assert np.array_equal(inter, oi) and np.array_equal(union, ou)


# ---------------------------------------------------------------------------------------------------------------------
# both kernel families against the oracle
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C", NARROW_C + WIDE_C)
@pytest.mark.parametrize("s", SHAPES)
@pytest.mark.parametrize("frac", [ONE_PIXEL, 0.1, 0.9])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("ign", [255, -100])
def test_ignore_vs_oracle(iic, cuda_device, ign, weighted, frac, s, C):
    rng = np.random.default_rng([C, len(s), int(weighted), 0 if frac == ONE_PIXEL else int(100 * frac), ign % 1000])
    lg = _logits(rng, (s[0], C) + tuple(s[1:]))
    lab = _labels(rng, s[0], C, s[1:], ign, frac)
    w = rng.uniform(0.2, 3.0, size=C).tolist() if weighted else None
    _check(_run(iic, cuda_device, lg, lab, ign, w, scale=3.0), _expected(lg, lab, ign, w), scale=3.0)


@pytest.mark.gpu
@pytest.mark.parametrize("C,ign", [(3, 1), (8, 0), (19, 0), (150, 149), (256, 255)])
def test_ignore_label_inside_class_range(iic, cuda_device, C, ign):
    """A class used as the ignore label: its pixels leave the loss and the Dice counts (its union still counts the
    kept pixels whose argmax is that class)."""
    rng = np.random.default_rng(C + ign)
    lg = _logits(rng, (2, C, 12, 20))
    lab = rng.integers(0, C, size=(2, 12, 20)).astype(np.int64)
    lab[0, :3] = ign                                    # make sure the class is present
    got = _run(iic, cuda_device, lg, lab, ign)
    want = _expected(lg, lab, ign)
    _check(got, want)
    assert (got[1].transpose(1, 0, 2, 3)[:, lab == ign] == 0).all()
    assert got[2][:, ign].sum() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 21])
@pytest.mark.parametrize("weighted", [False, True])
def test_absent_ignore_label_is_bit_identical(iic, cuda_device, C, weighted):
    rng = np.random.default_rng(70 + C)
    lg = _logits(rng, (3, C, 16, 24))
    lab = rng.integers(0, C, size=(3, 16, 24)).astype(np.int64)
    w = rng.uniform(0.2, 3.0, size=C).tolist() if weighted else None
    ref = _run(iic, cuda_device, lg, lab, None, w)
    for ign in (255, -100, C):
        got = _run(iic, cuda_device, lg, lab, ign, w)
        assert got[0] == ref[0]
        for a, b in zip(got[1:], ref[1:]):
            assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# edges
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 19, 150])
def test_one_sample_entirely_ignored(iic, cuda_device, C):
    rng = np.random.default_rng(80 + C)
    lg = _logits(rng, (3, C, 12, 20))
    lab = _labels(rng, 3, C, (12, 20), 255, 0.1)
    lab[1] = 255
    got = _run(iic, cuda_device, lg, lab, 255)
    _check(got, _expected(lg, lab, 255))
    assert not got[2][1].any() and not got[3][1].any()
    assert not got[1][1].any()


@pytest.mark.gpu
@pytest.mark.parametrize("C", [2, 5, 19, 256])
@pytest.mark.parametrize("weighted", [False, True])
def test_whole_batch_ignored(iic, cuda_device, C, weighted):
    rng = np.random.default_rng(90 + C)
    lg = _logits(rng, (2, C, 7, 9))
    lab = np.full((2, 7, 9), -100, np.int64)
    w = rng.uniform(0.2, 3.0, size=C).tolist() if weighted else None
    loss, grad, inter, union = _run(iic, cuda_device, lg, lab, -100, w)    # strict mode: a flag would raise here
    assert loss == 0.0
    assert not grad.any() and not inter.any() and not union.any()
    iic.raise_if_flagged(cuda_device)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 19])
def test_many_small_samples(iic, cuda_device, C):
    """300 samples of a 4 x 4 map: 300 rows of the (gx, outer) grid, each adding its own count."""
    rng = np.random.default_rng(300 + C)
    lg = _logits(rng, (300, C, 4, 4))
    lab = _labels(rng, 300, C, (4, 4), 255, 0.1)
    lab[7] = 255
    _check(_run(iic, cuda_device, lg, lab, 255), _expected(lg, lab, 255))


@pytest.mark.gpu
def test_one_large_map(iic, cuda_device):
    """One Cityscapes-sized map with 10 % void: every CTA of the (gx, 1) grid walks many tiles."""
    rng = np.random.default_rng(1024)
    lg = _logits(rng, (1, 19, 1024, 2048))
    lab = _labels(rng, 1, 19, (1024, 2048), 255, 0.1)
    _check(_run(iic, cuda_device, lg, lab, 255), _expected(lg, lab, 255))


# ---------------------------------------------------------------------------------------------------------------------
# other out-of-range labels next to the ignore label
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 21])
def test_bad_labels_with_ignore_label(iic, cuda_device, C):
    rng = np.random.default_rng(40 + C)
    lg = torch.from_numpy(_logits(rng, (2, C, 10, 12))).to(cuda_device)
    lab = torch.from_numpy(rng.integers(0, C, size=(2, 10, 12))).to(cuda_device)
    lab[0, 2, :] = 255
    lab[1, 3, 5] = -1
    with pytest.raises(AssertionError):
        iic.sup_kl_from_logits(lg.clone().requires_grad_(True), lab, ignore_index=255)
    iic.raise_if_flagged(cuda_device)
    with iic.check_mode("deferred"):
        c = lg.clone().requires_grad_(True)
        iic.sup_kl_from_logits(c, lab, ignore_index=255).backward()
        with pytest.raises(AssertionError):
            iic.raise_if_flagged(cuda_device)
    zero = (lab == 255) | (lab == -1)
    g = c.grad.permute(1, 0, 2, 3)
    assert float(g[:, zero].abs().max()) == 0.0
    assert bool((g[:, ~zero].abs().amax(0) > 0).all())
    # without the -1 the same map passes
    lab[1, 3, 5] = 0
    iic.sup_kl_from_logits(lg.clone().requires_grad_(True), lab, ignore_index=255).backward()


# ---------------------------------------------------------------------------------------------------------------------
# CUDA graph, determinism, torch cross-check
# ---------------------------------------------------------------------------------------------------------------------
def _step(iic, lp, lab, w):
    lp.grad = None
    loss, (inter, union) = iic.sup_kl_from_logits(lp, lab, weight=w, return_dice=True, ignore_index=255)
    loss.backward()
    return [loss.detach().clone(), inter.clone(), union.clone(), lp.grad.clone()]


@pytest.mark.gpu
@pytest.mark.parametrize("C", [4, 19, 150])
def test_graph_replay_with_changing_void(iic, cuda_device, C):
    """Forward + backward captured once; each replay sees labels rewritten in place with a different void fraction."""
    rng = np.random.default_rng(60 + C)
    B, H, W = 4, 64, 96
    lp = _dev(_logits(rng, (B, C, H, W)), cuda_device, grad=True)
    w = torch.from_numpy(rng.uniform(0.5, 2.0, size=C).astype(np.float32)).to(cuda_device)
    maps = [torch.from_numpy(_labels(rng, B, C, (H, W), 255, f)).to(cuda_device) for f in (0.0, 0.1, 0.9)]
    lab = maps[1].clone()
    with iic.check_mode("deferred"):
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            _step(iic, lp, lab, w)                              # warm-up on the capture stream (its workspaces)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        lp.grad = None
        with torch.cuda.graph(g, stream=side):
            out = _step(iic, lp, lab, w)
        for m in maps:
            lab.copy_(m)
            g.replay()
            torch.cuda.synchronize()
            got = [x.clone() for x in out]
            ref = _step(iic, lp, m, w)
            for x, y in zip(got, ref):
                assert torch.equal(x, y)
        iic.raise_if_flagged(cuda_device)
    # and the replays saw different denominators: the 90 % map's loss is the oracle's on its kept pixels
    lg = lp.detach().cpu().numpy()
    lab90 = maps[2].cpu().numpy()
    ol = _expected(lg, lab90, 255, w.cpu().tolist())[0]
    assert abs(float(ref[0]) - ol) <= LOSS_RTOL * abs(ol)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [3, 19, 150])
def test_repeat_determinism(iic, cuda_device, C):
    rng = np.random.default_rng(30 + C)
    lp = _dev(_logits(rng, (4, C, 64, 96)), cuda_device, grad=True)
    lab = torch.from_numpy(_labels(rng, 4, C, (64, 96), 255, 0.1)).to(cuda_device)
    w = torch.from_numpy(rng.uniform(0.5, 2.0, size=C).astype(np.float32)).to(cuda_device)
    a = _step(iic, lp, lab, w)
    b = _step(iic, lp, lab, w)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [19, 150])
def test_against_torch_cross_entropy(iic, cuda_device, C):
    """Without weights the loss is F.cross_entropy(ignore_index=255): the mean over the kept pixels."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(C)
    B, H, W = 4, 96, 128
    lg = (torch.randn(B, C, H, W, generator=g) * 2).to(cuda_device)
    lab = torch.randint(0, C, (B, H, W), generator=g)
    lab[torch.rand(B, H, W, generator=g) < 0.1] = 255
    lab = lab.to(cuda_device)
    a = lg.clone().requires_grad_(True)
    loss = iic.sup_kl_from_logits(a, lab, ignore_index=255)
    loss.backward()
    b = lg.double().requires_grad_(True)
    ref = F.cross_entropy(b, lab, ignore_index=255)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= LOSS_RTOL * abs(ref.item())
    assert relmax(a.grad.cpu().numpy(), b.grad.cpu().numpy()) <= GRAD_RTOL


# ---------------------------------------------------------------------------------------------------------------------
# argument checks (no GPU needed)
# ---------------------------------------------------------------------------------------------------------------------
def test_ignore_index_argument_checks():
    import iic_b200
    lg = torch.randn(2, 4, 8, 8, requires_grad=True)
    lab = torch.zeros(2, 8, 8, dtype=torch.int64)
    for bad in (True, False, 1.5, "255", torch.tensor(255)):
        with pytest.raises((TypeError, ValueError)):
            iic_b200.sup_kl_from_logits(lg, lab, ignore_index=bad)
    with pytest.raises(ValueError):
        iic_b200.sup_kl_from_logits(lg, lab, ignore_index=2 ** 63)
    for ign in (255, -100, np.int64(255)):
        with pytest.raises(Exception) as ei:                # CPU tensors are refused: no CPU fallback
            iic_b200.sup_kl_from_logits(lg, lab, ignore_index=ign)
        assert "CPU" in str(ei.value) or "CUDA" in str(ei.value)
