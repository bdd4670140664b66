"""The wide-class path (9 <= C <= 256) of the UDA, supervised and flip-aligned losses against the fp64 oracle.

Bounds as everywhere in the suite: loss 1e-5 relative, gradient 1e-4 max-norm relative.  The C values cover every
slice width of the kernels (ceil(C / 8) rounded up to 2, 4, 8, 16 or 32 channels per warp) on both sides of each
boundary; the shapes select both pixel-group widths (inner % 4 == 0 -> 4 pixels per lane, else 1) and end on a partial
tile of 32 groups.
"""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, relmax

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-5
GRAD_RTOL = 1e-4
WIDE_C = [9, 16, 17, 19, 21, 32, 33, 64, 65, 128, 129, 150, 256]
# inner = 240 (% 4 == 0: 60 groups of 4, the second tile partial), inner = 63 (% 4 != 0), and a 2-D (N, C) input
UDA_SHAPES = [(2, 12, 20), (3, 7, 9), (70,)]


@pytest.fixture(scope="module")
def iic(cuda_device):
    import iic_b200
    return iic_b200


def _shape(C, s):
    return (s[0], C) + tuple(s[1:])


def _logits(rng, shape, scale=2.0):
    return (rng.standard_normal(shape) * scale).astype(np.float32)


def _dev(a, dev, grad=False):
    t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    return t.requires_grad_(True) if grad else t


# ---------------------------------------------------------------------------------------------------------------------
# UDA: MSELoss / KL_div on probabilities, uda_from_logits
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDE_C)
@pytest.mark.parametrize("s", UDA_SHAPES)
@pytest.mark.parametrize("kind", ["mse", "kl"])
def test_uda_wide_vs_oracle(iic, cuda_device, kind, s, C):
    shape = _shape(C, s)
    rng = np.random.default_rng(1000 + C + 7 * len(s))
    lp, lt = _logits(rng, shape), _logits(rng, shape)
    p, t = O.softmax(lp).astype(np.float32), O.softmax(lt).astype(np.float32)
    fn = O.mse_loss if kind == "mse" else O.kl_div
    pd = _dev(p, cuda_device, grad=True)
    crit = iic.MSELoss() if kind == "mse" else iic.KL_div(verbose=False)
    loss = crit(pd, _dev(t, cuda_device))
    (3.0 * loss).backward()
    ol, og = fn(p, t, with_grads=True)
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(pd.grad.cpu().numpy(), 3.0 * og) <= GRAD_RTOL
    ld = _dev(lp, cuda_device, grad=True)
    lf = iic.uda_from_logits(ld, _dev(lt, cuda_device), kind)
    lf.backward()
    p64, t64 = O.softmax(lp), O.softmax(lt)
    ol2, og2 = fn(p64, t64, with_grads=True)
    assert abs(lf.item() - ol2) <= LOSS_RTOL * abs(ol2)
    assert relmax(ld.grad.cpu().numpy(), O.softmax_backward(p64, og2)) <= GRAD_RTOL


@pytest.mark.parametrize("s", UDA_SHAPES)
def test_kl_div_class_weights_c19(iic, cuda_device, s):
    C = 19
    rng = np.random.default_rng(19 + len(s))
    shape = _shape(C, s)
    p = O.softmax(_logits(rng, shape)).astype(np.float32)
    t = O.softmax(_logits(rng, shape)).astype(np.float32)
    w = rng.uniform(0.2, 3.0, size=C).tolist()
    pd = _dev(p, cuda_device, grad=True)
    loss = iic.KL_div(weight=w, verbose=False)(pd, _dev(t, cuda_device))
    loss.backward()
    ol, og = O.kl_div(p, t, weight=w, with_grads=True)
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(pd.grad.cpu().numpy(), og) <= GRAD_RTOL


def test_simplex_check_wide(iic, cuda_device):
    C = 12
    rng = np.random.default_rng(12)
    p = O.softmax(_logits(rng, (2, C, 8, 12))).astype(np.float32)
    t = O.softmax(_logits(rng, (2, C, 8, 12))).astype(np.float32)
    good = p.copy()
    p[1, :, 5, 7] *= 1.01                                   # one pixel off the simplex
    with pytest.raises(AssertionError):
        iic.KL_div(verbose=False)(_dev(p, cuda_device, grad=True), _dev(t, cuda_device))
    with iic.check_mode("deferred"):
        iic.KL_div(verbose=False)(_dev(p, cuda_device, grad=True), _dev(t, cuda_device))
        with pytest.raises(AssertionError):
            iic.raise_if_flagged(cuda_device)
    iic.raise_if_flagged(cuda_device)                     # clean again
    iic.KL_div(verbose=False)(_dev(good, cuda_device, grad=True), _dev(t, cuda_device))   # a simplex input passes


# ---------------------------------------------------------------------------------------------------------------------
# supervised: KL against the one-hot label, class weights, Dice counts
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", WIDE_C)
@pytest.mark.parametrize("s", [(2, 12, 20), (3, 7, 9)])
@pytest.mark.parametrize("weighted", [False, True])
def test_supervised_wide_vs_oracle(iic, cuda_device, weighted, s, C):
    shape = _shape(C, s)
    rng = np.random.default_rng(2000 + C + len(s) + 3 * weighted)
    lg = _logits(rng, shape)
    lab = rng.integers(0, C, size=shape[:1] + shape[2:]).astype(np.int64)
    w = rng.uniform(0.2, 3.0, size=C).tolist() if weighted else None
    ld = _dev(lg, cuda_device, grad=True)
    loss, (inter, union) = iic.sup_kl_from_logits(ld, _dev(lab, cuda_device), weight=w, return_dice=True)
    (3.0 * loss).backward()
    ol, og = O.sup_kl_from_logits(lg, lab, weight=w, with_grads=True)
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(ld.grad.cpu().numpy(), 3.0 * og) <= GRAD_RTOL
    oi, ou = O.dice_counts(lg, lab)
    assert np.array_equal(inter.cpu().numpy(), oi) and np.array_equal(union.cpu().numpy(), ou)


@pytest.mark.parametrize("C", [19, 150])
def test_supervised_dice_ties_first_index_wins(iic, cuda_device, C):
    """Logits quantised to a few values, so most pixels have an exactly tied maximum, often in different warps."""
    rng = np.random.default_rng(C)
    lg = rng.integers(-2, 2, size=(2, C, 9, 16)).astype(np.float32)
    lab = rng.integers(0, C, size=(2, 9, 16)).astype(np.int64)
    loss, (inter, union) = iic.sup_kl_from_logits(_dev(lg, cuda_device, grad=True), _dev(lab, cuda_device),
                                                  return_dice=True)
    oi, ou = O.dice_counts(lg, lab)
    assert np.array_equal(inter.cpu().numpy(), oi) and np.array_equal(union.cpu().numpy(), ou)
    assert abs(loss.item() - O.sup_kl_from_logits(lg, lab)) <= LOSS_RTOL * abs(O.sup_kl_from_logits(lg, lab))


@pytest.mark.parametrize("bad_label", [-1, 21])
def test_supervised_wide_bad_labels(iic, cuda_device, bad_label):
    C = 21
    rng = np.random.default_rng(21)
    lg = torch.from_numpy(_logits(rng, (2, C, 10, 12))).to(cuda_device)
    lab = torch.from_numpy(rng.integers(0, C, size=(2, 10, 12))).to(cuda_device)
    lab[1, 3, 5] = bad_label
    with pytest.raises(AssertionError):
        iic.sup_kl_from_logits(lg.clone().requires_grad_(True), lab)
    with iic.check_mode("deferred"):
        c = lg.clone().requires_grad_(True)
        iic.sup_kl_from_logits(c, lab).backward()
        assert float(c.grad[1, :, 3, 5].abs().max()) == 0.0
        assert float(c.grad[1, :, 3, 6].abs().max()) > 0.0
        with pytest.raises(AssertionError):
            iic.raise_if_flagged(cuda_device)
    iic.raise_if_flagged(cuda_device)


# ---------------------------------------------------------------------------------------------------------------------
# UDA through the per-sample flips
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [9, 19, 64, 150, 256])
@pytest.mark.parametrize("HW", [(12, 20), (7, 9)])
@pytest.mark.parametrize("kind", ["mse", "kl"])
def test_flip_wide_vs_oracle(iic, cuda_device, kind, HW, C):
    B = 4
    shape = (B, C) + HW
    rng = np.random.default_rng(3000 + C + HW[1])
    ls, lt = _logits(rng, shape), _logits(rng, shape)
    flags = np.arange(B, dtype=np.uint8) % 4                 # none / H / W / both
    sd = _dev(ls, cuda_device, grad=True)
    loss = iic.uda_from_logits(sd, _dev(lt, cuda_device), kind, teacher_flips=torch.from_numpy(flags))
    (2.0 * loss).backward()
    ol, og = O.uda_from_logits_flipped(ls, lt, flags, kind, with_grads=True)
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(sd.grad.cpu().numpy(), 2.0 * og) <= GRAD_RTOL


# ---------------------------------------------------------------------------------------------------------------------
# dispatch, limits, grid edges, determinism, CUDA graphs
# ---------------------------------------------------------------------------------------------------------------------
def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def _run_all_families(iic, dev, C):
    rng = np.random.default_rng(C)
    shape = (2, C, 8, 12)
    lp = _dev(_logits(rng, shape), dev, grad=True)
    lt = _dev(_logits(rng, shape), dev)
    iic.uda_from_logits(lp, lt, "kl").backward()
    iic.uda_from_logits(lp, lt, "mse", teacher_flips=torch.tensor([1, 2], dtype=torch.uint8)).backward()
    lab = _dev(rng.integers(0, C, size=(2, 8, 12)), dev)
    iic.sup_kl_from_logits(lp, lab).backward()


def test_dispatch_by_class_count(iic, cuda_device):
    names8 = _kernel_names(lambda: _run_all_families(iic, cuda_device, 8))
    names9 = _kernel_names(lambda: _run_all_families(iic, cuda_device, 9))
    for fam in ("uda_fwd", "uda_bwd", "sup_fwd", "sup_bwd", "uda_flip_fwd", "uda_flip_bwd"):
        assert any(f"{fam}_" in n and "wide" not in n for n in names8), (fam, names8)
        assert not any(f"{fam}_wide_kernel" in n for n in names8), (fam, names8)
        assert any(f"{fam}_wide_kernel" in n for n in names9), (fam, names9)


def test_class_limit(iic, cuda_device):
    rng = np.random.default_rng(257)
    x = _dev(_logits(rng, (2, 257, 4, 4)), cuda_device, grad=True)
    y = _dev(_logits(rng, (2, 257, 4, 4)), cuda_device)
    lab = _dev(rng.integers(0, 257, size=(2, 4, 4)), cuda_device)
    with pytest.raises(RuntimeError, match="256"):
        iic.uda_from_logits(x, y, "mse")
    with pytest.raises(RuntimeError, match="256"):
        iic.uda_from_logits(x, y, "kl", teacher_flips=torch.tensor([0, 3], dtype=torch.uint8))
    with pytest.raises(RuntimeError, match="256"):
        iic.sup_kl_from_logits(x, lab)


def test_grid_edges(iic, cuda_device):
    # one sample with a large map: every CTA of the (gx, 1) grid walks many tiles
    rng = np.random.default_rng(7)
    lg = _logits(rng, (1, 21, 512, 1020))
    lab = rng.integers(0, 21, size=(1, 512, 1020)).astype(np.int64)
    ld = _dev(lg, cuda_device, grad=True)
    loss, (inter, union) = iic.sup_kl_from_logits(ld, _dev(lab, cuda_device), return_dice=True)
    loss.backward()
    ol, og = O.sup_kl_from_logits(lg, lab, with_grads=True)
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(ld.grad.cpu().numpy(), og) <= GRAD_RTOL
    oi, ou = O.dice_counts(lg, lab)
    assert np.array_equal(inter.cpu().numpy(), oi) and np.array_equal(union.cpu().numpy(), ou)
    lt = _logits(rng, (1, 21, 512, 1020))
    ud = _dev(lg, cuda_device, grad=True)
    ul = iic.uda_from_logits(ud, _dev(lt, cuda_device), "kl", teacher_flips=torch.tensor([3], dtype=torch.uint8))
    ul.backward()
    ol, og = O.uda_from_logits_flipped(lg, lt, np.array([3], np.uint8), "kl", with_grads=True)
    assert abs(ul.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(ud.grad.cpu().numpy(), og) <= GRAD_RTOL
    # 300 samples of a 4 x 4 map: one partial tile per sample, 300 rows of the grid
    B, C = 300, 19
    lg = _logits(rng, (B, C, 4, 4))
    lt = _logits(rng, (B, C, 4, 4))
    lab = rng.integers(0, C, size=(B, 4, 4)).astype(np.int64)
    ld = _dev(lg, cuda_device, grad=True)
    loss, (inter, union) = iic.sup_kl_from_logits(ld, _dev(lab, cuda_device), return_dice=True)
    loss.backward()
    ol, og = O.sup_kl_from_logits(lg, lab, with_grads=True)
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol)
    assert relmax(ld.grad.cpu().numpy(), og) <= GRAD_RTOL
    oi, ou = O.dice_counts(lg, lab)
    assert np.array_equal(inter.cpu().numpy(), oi) and np.array_equal(union.cpu().numpy(), ou)
    flags = (np.arange(B) % 4).astype(np.uint8)
    for kind in ("mse", "kl"):
        sd = _dev(lg, cuda_device, grad=True)
        ul = iic.uda_from_logits(sd, _dev(lt, cuda_device), kind, teacher_flips=torch.from_numpy(flags))
        ul.backward()
        ol, og = O.uda_from_logits_flipped(lg, lt, flags, kind, with_grads=True)
        assert abs(ul.item() - ol) <= LOSS_RTOL * abs(ol)
        assert relmax(sd.grad.cpu().numpy(), og) <= GRAD_RTOL
        ud = _dev(lg, cuda_device, grad=True)
        ul = iic.uda_from_logits(ud, _dev(lt, cuda_device), kind)
        ul.backward()
        p64, t64 = O.softmax(lg), O.softmax(lt)
        ol, og = (O.mse_loss if kind == "mse" else O.kl_div)(p64, t64, with_grads=True)
        assert abs(ul.item() - ol) <= LOSS_RTOL * abs(ol)
        assert relmax(ud.grad.cpu().numpy(), O.softmax_backward(p64, og)) <= GRAD_RTOL


def _step(iic, lp, lt, lab, flags, w):
    """UDA (plain and through the flips) + supervised with Dice; returns the losses, counts and gradients."""
    lp.grad = None
    u1 = iic.uda_from_logits(lp, lt, "kl")
    u2 = iic.uda_from_logits(lp, lt, "mse", teacher_flips=flags)
    s, (inter, union) = iic.sup_kl_from_logits(lp, lab, weight=w, return_dice=True)
    (u1 + u2 + s).backward()
    return [u1.detach().clone(), u2.detach().clone(), s.detach().clone(), inter.clone(), union.clone(),
            lp.grad.clone()]


@pytest.mark.parametrize("C", [19, 150])
def test_wide_determinism_and_graph_replay(iic, cuda_device, C):
    rng = np.random.default_rng(50 + C)
    shape = (4, C, 64, 96)
    lp = _dev(_logits(rng, shape), cuda_device, grad=True)
    lt = _dev(_logits(rng, shape), cuda_device)
    lab = _dev(rng.integers(0, C, size=(4, 64, 96)), cuda_device)
    flags = torch.tensor([0, 1, 2, 3], dtype=torch.uint8, device=cuda_device)
    w = torch.from_numpy(rng.uniform(0.5, 2.0, size=C).astype(np.float32)).to(cuda_device)
    with iic.check_mode("deferred"):
        a = _step(iic, lp, lt, lab, flags, w)
        b = _step(iic, lp, lt, lab, flags, w)
        for x, y in zip(a, b):
            assert torch.equal(x, y)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            _step(iic, lp, lt, lab, flags, w)                 # warm-up on the capture stream (its workspaces)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        lp.grad = None
        with torch.cuda.graph(g, stream=side):
            out = _step(iic, lp, lt, lab, flags, w)
        for _ in range(2):
            g.replay()
            torch.cuda.synchronize()
            for x, y in zip(out, a):
                assert torch.equal(x, y)
        iic.raise_if_flagged(cuda_device)


def test_cityscapes_step_against_torch(iic, cuda_device):
    """A Cityscapes-shaped step against the eager torch composition of the reference's formulas."""
    import torch.nn.functional as F
    B, C, H, W = 4, 19, 128, 256
    g = torch.Generator().manual_seed(19)
    s_log = (torch.randn(B, C, H, W, generator=g) * 2).to(cuda_device)
    t_log = (torch.randn(B, C, H, W, generator=g) * 2).to(cuda_device)
    lab = torch.randint(0, C, (B, H, W), generator=g).to(cuda_device)
    w = torch.rand(C, generator=g) + 0.5

    a = s_log.clone().requires_grad_(True)
    u = iic.uda_from_logits(a, t_log, "kl")
    s, (inter, union) = iic.sup_kl_from_logits(a, lab, weight=w, return_dice=True)
    (u + s).backward()

    b = s_log.double().requires_grad_(True)
    p, t = b.softmax(1), t_log.double().softmax(1)
    eps = 1e-16
    u_ref = (-t * torch.log((p + eps) / (t + eps))).sum(1).mean()
    onehot = F.one_hot(lab, C).permute(0, 3, 1, 2).double()
    wn = (w / w.sum() * C).double().to(cuda_device).view(1, C, 1, 1)
    s_ref = (-onehot * torch.log((p + eps) / (onehot + eps)) * wn).sum(1).mean()
    (u_ref + s_ref).backward()
    pred = F.one_hot(b.detach().max(1)[1], C).permute(0, 3, 1, 2)
    oh = F.one_hot(lab, C).permute(0, 3, 1, 2)
    assert abs(u.item() - u_ref.item()) <= LOSS_RTOL * abs(u_ref.item())
    assert abs(s.item() - s_ref.item()) <= LOSS_RTOL * abs(s_ref.item())
    assert relmax(a.grad.cpu().numpy(), b.grad.cpu().numpy()) <= GRAD_RTOL
    assert torch.equal(inter, (pred * oh).sum((2, 3))) and torch.equal(union, (pred + oh).sum((2, 3)))
