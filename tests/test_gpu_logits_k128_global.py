"""The cluster head's softmax fused into the wide heads' local IIC term (K = 128, padding 1: the stats pass, the
from-logits tensor-core joint and backward) and into the global IIC terms (the finish launch normalises the (N, K) logit
rows; global_backward_kernel<true> applies the softmax adjoint), reached through IIDSegmentationSmallPathLoss.from_logits,
IIDLoss.from_logits and iic_losses(from_logits=True).

Losses and LOGIT gradients are compared with the fp64 oracle chained through its own softmax (O.softmax,
O.softmax_backward with T) at the project's bounds: loss 1e-5 relative, gradients 1e-4 max-norm relative.  Which
kernels ran is read from torch.profiler (full names, so that the from-logits instantiations <true> are told apart)."""
import contextlib
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
K = 128


@pytest.fixture(scope="module")
def iic(cuda_device):
    import iic_b200
    return iic_b200


@contextlib.contextmanager
def options(iic, **opts):
    old = {k: iic._lib.set_option(k, v) for k, v in opts.items()}
    try:
        yield
    finally:
        for k, v in old.items():
            iic._lib.set_option(k, v)


def logit_views(rng, B, K, H, W, scale=1.0):
    """Two correlated logit maps (a coarse shared field plus independent noise), as a cluster head gives for two views."""
    base = rng.standard_normal((B, K, -(-H // 4), -(-W // 4))).repeat(4, axis=2).repeat(4, axis=3)[:, :, :H, :W] * 3
    l1 = ((base + 0.5 * rng.standard_normal((B, K, H, W))) * scale).astype(np.float32)
    l2 = ((base + 0.5 * rng.standard_normal((B, K, H, W))) * scale).astype(np.float32)
    return l1, l2


def oracle(l1, l2, pad, T, up=1.0):
    p1, p2 = O.softmax(l1, 1, T), O.softmax(l2, 1, T)
    ol, gp1, gp2 = O.iid_segmentation_small_path_loss(p1, p2, pad, 4096, with_grads=True)
    return ol, up * O.softmax_backward(p1, gp1, 1, T), up * O.softmax_backward(p2, gp2, 1, T)


def launched(fn):
    """Full names of every CUDA kernel one call of fn launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if getattr(e, "device_type", None) is not None and "(" in e.name]


def fused_names(names):
    return {"stats": any("local_logit_stats_kernel" in n for n in names),
            "tc": any("local_joint_tc_kernel<true>" in n for n in names),
            "bwd": any("local_bwd_tc_kernel<true>" in n for n in names),
            "softmax": any("softmax" in n.lower() for n in names)}


def run_from_logits(iic, dev, l1, l2, pad, T, up=0.37):
    a = torch.from_numpy(l1).to(dev).requires_grad_(True)
    b = torch.from_numpy(l2).to(dev).requires_grad_(True)
    loss = iic.IIDSegmentationSmallPathLoss(padding=pad, patch_size=4096).from_logits(a, b, T=T)
    (up * loss).backward()
    return loss.item(), a.grad.cpu().numpy(), b.grad.cpu().numpy()


def check(loss, ga, gb, ol, og1, og2):
    assert abs(loss - ol) <= LOSS_RTOL * max(abs(ol), 0.05), (loss, ol)
    ex, ey = relmax(ga, og1), relmax(gb, og2)
    print(f"loss rel {abs(loss - ol) / max(abs(ol), 1e-30):.2e}  grad relmax {max(ex, ey):.2e}")
    assert ex <= GRAD_RTOL and ey <= GRAD_RTOL, (ex, ey)


# ---------------------------------------------------------------------------------------------------
# K = 128 against the oracle: temperature x (normal, sharply peaked logits), and the kernels' edges
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("peaked", [False, True])
@pytest.mark.parametrize("T", [1.0, 0.1])
def test_k128_from_logits_vs_oracle(iic, cuda_device, T, peaked):
    rng = np.random.default_rng(int(10 * T) + 7 * peaked)
    B, H, W = 2, 20, 48
    # peaked: logits scaled so that l / T spans hundreds at T = 0.1, p one-hot up to fp32
    l1, l2 = logit_views(rng, B, K, H, W, scale=8.0 if peaked else 1.0)
    a = torch.from_numpy(l1).to(cuda_device)
    assert iic.ops.from_logits_covered(a, a, 1)
    names = launched(lambda: run_from_logits(iic, cuda_device, l1, l2, 1, T))
    f = fused_names(names)
    assert f["stats"] and f["tc"] and f["bwd"] and not f["softmax"], names
    loss, ga, gb = run_from_logits(iic, cuda_device, l1, l2, 1, T)
    check(loss, ga, gb, *oracle(l1, l2, 1, T, 0.37))


@pytest.mark.parametrize("B,H,W", [
    (1, 12, 32),          # B = 1
    (2, 13, 32),          # odd H: the backward's last row pair has one row
    (2, 10, 16),          # W = 16: one k-block per row, the joint's x box reaches past both map edges
    (1, 9, 240),          # W = 240: two 128-pixel tiles in the backward, a TMA box of 248 columns
    (3, 112, 112),        # long accumulation runs: many TMEM segments per joint CTA, many items per backward CTA
])
def test_k128_from_logits_edges(iic, cuda_device, B, H, W):
    rng = np.random.default_rng(B * 7 + H * 13 + W)
    l1, l2 = logit_views(rng, B, K, H, W)
    names = launched(lambda: run_from_logits(iic, cuda_device, l1, l2, 1, 0.5))
    f = fused_names(names)
    assert f["stats"] and f["tc"] and f["bwd"] and not f["softmax"], names
    loss, ga, gb = run_from_logits(iic, cuda_device, l1, l2, 1, 0.5)
    check(loss, ga, gb, *oracle(l1, l2, 1, 0.5, 0.37))


def test_k128_from_logits_repeatable(iic, cuda_device):
    """Two identical calls give bit-identical loss and gradients."""
    rng = np.random.default_rng(5)
    l1, l2 = logit_views(rng, 2, K, 24, 144)
    r1 = run_from_logits(iic, cuda_device, l1, l2, 1, 0.1)
    r2 = run_from_logits(iic, cuda_device, l1, l2, 1, 0.1)
    assert r1[0] == r2[0]
    assert np.array_equal(r1[1], r2[1]) and np.array_equal(r1[2], r2[2])


# ---------------------------------------------------------------------------------------------------
# channel blocks of one (2B, 2*128, H, W) head output: gradients land in their blocks, nothing else is written
# ---------------------------------------------------------------------------------------------------
def test_k128_blocks_of_head_output_and_sentinels(iic, cuda_device):
    S, B, H, W, T = 2, 2, 12, 32, 0.5
    rng = np.random.default_rng(12)
    full = rng.standard_normal((2 * B, S * K, H, W)).astype(np.float32) * 2
    t = torch.from_numpy(full).to(cuda_device).requires_grad_(True)
    halves = torch.chunk(t, 2, 0)                                     # the epocher's (view 1, view 2) split
    crit = iic.IIDSegmentationSmallPathLoss(padding=1, patch_size=4096)
    a, b = halves[0][:, K:], halves[1][:, K:]                         # sub-head 1 only
    crit.from_logits(a, b, T=T).backward()
    g = t.grad.cpu().numpy()
    _, og1, og2 = oracle(full[:B, K:], full[B:, K:], 1, T)
    assert relmax(g[:B, K:], og1) <= GRAD_RTOL and relmax(g[B:, K:], og2) <= GRAD_RTOL
    assert not g[:, :K].any()

    # the raw backward entry point writing into channel-block views of sentinel-filled tensors
    lx = torch.from_numpy(full[:B]).to(cuda_device).contiguous()
    ly = torch.from_numpy(full[B:]).to(cuda_device).contiguous()
    a, b = lx[:, :K], ly[:, :K]
    term = iic.ops.LocalTerm(a, b, None, 1, (H, W), (H, W), 1.0, logits=True, inv_temperature=1.0 / T)
    (r,) = iic.ops._finish_terms([term], False)
    assert r["stats"] is not None
    GX = torch.full((B, S * K, H, W), 7.25, device=cuda_device)
    GY = torch.full((B, S * K, H, W), -3.5, device=cuda_device)
    gx, gy = GX[:, :K], GY[:, :K]
    gx.fill_(float("nan"))
    gy.fill_(float("nan"))
    iic.ops._local_backward_logits_stats_into(a, b, r["stats"], r["Wx"], r["Wy"], torch.ones((), device=cuda_device), 1,
                                             1.0 / T, gx, gy)
    _, og1, og2 = oracle(full[:B, :K], full[B:, :K], 1, T)
    assert relmax(gx.cpu().numpy(), og1) <= GRAD_RTOL and relmax(gy.cpu().numpy(), og2) <= GRAD_RTOL
    assert bool((GX[:, K:] == 7.25).all()) and bool((GY[:, K:] == -3.5).all())


# ---------------------------------------------------------------------------------------------------
# K = 128 dispatch: covered shapes run the fused kernels and no torch softmax; the query agrees with what ran
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,H,W,pad,opts,fused", [
    (2, 16, 64, 1, {}, True),
    (2, 16, 40, 1, {}, False),                    # W % 16 != 0
    (1, 8, 256, 1, {}, False),                    # W > 248
    (2, 16, 32, 3, {}, False),                    # padding 3
    (2, 16, 64, 1, {"no_tc": 1}, False),          # tensor cores switched off
    (2, 16, 64, 1, {"no_tma": 1}, False),         # TMA switched off
])
def test_k128_query_matches_what_ran(iic, cuda_device, B, H, W, pad, opts, fused):
    rng = np.random.default_rng(B + H + W + pad)
    l1, l2 = logit_views(rng, B, K, H, W)
    with options(iic, **opts):
        a = torch.from_numpy(l1).to(cuda_device)
        b = torch.from_numpy(l2).to(cuda_device)
        assert iic.ops.from_logits_covered(a, b, pad) == fused
        names = launched(lambda: run_from_logits(iic, cuda_device, l1, l2, pad, 1.0))
        loss, ga, gb = run_from_logits(iic, cuda_device, l1, l2, pad, 1.0)
    f = fused_names(names)
    if fused:
        assert f["stats"] and f["tc"] and f["bwd"] and not f["softmax"], names
    else:
        assert not (f["stats"] or f["tc"] or f["bwd"]) and f["softmax"], names
    if pad == 1 and W <= 64:
        check(loss, ga, gb, *oracle(l1, l2, pad, 1.0, 0.37))


# ---------------------------------------------------------------------------------------------------
# global terms from logits
# ---------------------------------------------------------------------------------------------------
def global_oracle(l1, l2, T, lamb, gl, gnl, gP):
    p1, p2 = O.softmax(l1, 1, T), O.softmax(l2, 1, T)
    loss, loss_nl, P = O.iid_loss(p1, p2, lamb)
    dx, dy = O.iid_loss_grads(p1, p2, lamb, gl, gnl, gP)
    return loss, loss_nl, P, O.softmax_backward(p1, dx, 1, T), O.softmax_backward(p2, dy, 1, T)


def run_global(iic, dev, l1, l2, T, lamb, gl, gnl, gP):
    a = torch.from_numpy(l1).to(dev).requires_grad_(True)
    b = torch.from_numpy(l2).to(dev).requires_grad_(True)
    loss, loss_nl, P = iic.IIDLoss(lamb=lamb).from_logits(a, b, T=T)
    obj = gl * loss + gnl * loss_nl
    if gP is not None:
        obj = obj + (P * torch.from_numpy(gP).to(dev)).sum()
    obj.backward()
    return float(loss), float(loss_nl), P.detach().cpu().numpy(), a.grad.cpu().numpy(), b.grad.cpu().numpy()


def check_global(res, ref):
    loss, loss_nl, P, ga, gb = res
    ol, onl, oP, og1, og2 = ref
    assert abs(loss - ol) <= LOSS_RTOL * max(abs(ol), 0.05), (loss, ol)
    assert abs(loss_nl - onl) <= LOSS_RTOL * max(abs(onl), 0.05), (loss_nl, onl)
    assert relmax(P, oP) <= 1e-5
    ex, ey = relmax(ga, og1), relmax(gb, og2)
    print(f"loss rel {abs(loss - ol) / max(abs(ol), 1e-30):.2e}  grad relmax {max(ex, ey):.2e}")
    assert ex <= GRAD_RTOL and ey <= GRAD_RTOL, (ex, ey)


@pytest.mark.parametrize("out", ["loss", "loss_no_lamb", "P"])
@pytest.mark.parametrize("T", [0.1, 1.0, 2.0])
@pytest.mark.parametrize("N,KG", [(4, 10), (64, 20), (10, 128), (4096, 10)])
def test_global_from_logits_vs_oracle(iic, cuda_device, N, KG, T, out):
    rng = np.random.default_rng(N + KG + int(10 * T) + len(out))
    shared = rng.standard_normal((N, KG)) * 2
    l1 = (shared + 0.7 * rng.standard_normal((N, KG))).astype(np.float32)
    l2 = (shared + 0.7 * rng.standard_normal((N, KG))).astype(np.float32)
    lamb = 1.3
    gl, gnl, gP = {"loss": (0.7, 0.0, None), "loss_no_lamb": (0.0, 1.1, None),
                   "P": (0.0, 0.0, rng.standard_normal((KG, KG)).astype(np.float32))}[out]
    names = launched(lambda: run_global(iic, cuda_device, l1, l2, T, lamb, gl, gnl, gP))
    assert sum("finish_kernel" in n for n in names) == 1 and not any("softmax" in n.lower() for n in names), names
    assert any("global_backward_kernel<true>" in n for n in names), names
    check_global(run_global(iic, cuda_device, l1, l2, T, lamb, gl, gnl, gP), global_oracle(l1, l2, T, lamb, gl, gnl, gP))


def test_global_from_logits_repeatable(iic, cuda_device):
    rng = np.random.default_rng(9)
    l1 = rng.standard_normal((300, 128)).astype(np.float32)
    l2 = rng.standard_normal((300, 128)).astype(np.float32)
    r1 = run_global(iic, cuda_device, l1, l2, 0.5, 1.0, 1.0, 0.5, None)
    r2 = run_global(iic, cuda_device, l1, l2, 0.5, 1.0, 1.0, 0.5, None)
    assert r1[0] == r2[0] and r1[1] == r2[1]
    for u, v in zip(r1[2:], r2[2:]):
        assert np.array_equal(u, v)


def test_global_from_logits_fallback_past_4096_rows(iic, cuda_device):
    """N = 4097 is not covered: the softmax runs first and the result still matches."""
    rng = np.random.default_rng(4097)
    l1 = rng.standard_normal((4097, 10)).astype(np.float32)
    l2 = (l1 + 0.5 * rng.standard_normal((4097, 10))).astype(np.float32)
    a = torch.from_numpy(l1).to(cuda_device)
    assert not iic.ops.global_logits_covered(a, a)
    names = launched(lambda: run_global(iic, cuda_device, l1, l2, 0.5, 1.0, 1.0, 0.0, None))
    assert any("softmax" in n.lower() for n in names) and not any("global_backward_kernel<true>" in n for n in names)
    check_global(run_global(iic, cuda_device, l1, l2, 0.5, 1.0, 1.0, 0.0, None),
                 global_oracle(l1, l2, 0.5, 1.0, 1.0, 0.0, None))


def test_global_from_logits_cluster_head_rows(iic, cuda_device):
    """Strided (N, K) rows: the sub-head views ClusterHead.logits() returns for a batch of both augmented views; each
    gradient lands in its block of the head output, through to the head's weights, as for the softmax path."""
    from iic_b200.trainer._utils import ClusterHead
    torch.manual_seed(0)
    S, KG, N, T = 3, 10, 16, 0.5
    head = ClusterHead(input_dim=32, num_clusters=KG, num_subheads=S, T=T).to(cuda_device)
    feats = torch.randn(2 * N, 32, 4, 4, device=cuda_device)

    def total(from_logits):
        head.zero_grad()
        outs = head.logits(feats) if from_logits else head(feats)
        loss = 0.0
        crit = iic.IIDLoss()
        for o in outs:
            a, b = torch.chunk(o, 2, 0)
            loss = loss + (crit.from_logits(a, b, T=T)[0] if from_logits else crit(a, b)[0])
        loss.backward()
        return float(loss), [p.grad.detach().cpu().numpy().copy() for p in head.parameters() if p.grad is not None]

    outs = head.logits(feats)
    assert any(o.stride(0) != o.shape[1] for o in outs) or len(outs) == 1   # views into the (2N, S*K) head output
    l_f, g_f = total(True)
    l_p, g_p = total(False)
    assert abs(l_f - l_p) <= LOSS_RTOL * max(abs(l_p), 0.05), (l_f, l_p)
    assert len(g_f) == len(g_p) > 0
    for u, v in zip(g_f, g_p):
        assert relmax(u, v) <= GRAD_RTOL

    # against the oracle on the rows themselves
    with torch.no_grad():
        lo = [o.detach().cpu().numpy() for o in head.logits(feats)]
    for s in range(S):
        l1, l2 = lo[s][:N], lo[s][N:]
        a = torch.from_numpy(np.ascontiguousarray(l1)).to(cuda_device)
        b = torch.from_numpy(np.ascontiguousarray(l2)).to(cuda_device)
        loss, loss_nl, P = iic.IIDLoss().from_logits(a, b, T=T)
        assert abs(float(loss) - global_oracle(l1, l2, T, 1.0, 1.0, 0.0, None)[0]) <= LOSS_RTOL * 0.05 + LOSS_RTOL * abs(float(loss))


def test_semi_seg_wrapper_returns_loss_only(iic, cuda_device):
    from iic_b200.semi_seg._utils import IIDLoss as WrappedIIDLoss
    rng = np.random.default_rng(1)
    a = torch.from_numpy(rng.standard_normal((8, 10)).astype(np.float32)).to(cuda_device).requires_grad_(True)
    b = torch.from_numpy(rng.standard_normal((8, 10)).astype(np.float32)).to(cuda_device).requires_grad_(True)
    r = WrappedIIDLoss().from_logits(a, b, T=0.5)
    assert isinstance(r, torch.Tensor) and r.dim() == 0
    assert float(r) == float(iic.IIDLoss().from_logits(a, b, T=0.5)[0])


# ---------------------------------------------------------------------------------------------------
# the batched API: 5 global and 5 local terms from logits in ONE finish launch, no softmax kernel
# ---------------------------------------------------------------------------------------------------
def test_iic_losses_from_logits_global_and_k128(iic, cuda_device):
    S, B, KG, H, W, T = 5, 4, 10, 8, 32, 0.5
    rng = np.random.default_rng(2027)
    glob_rows = (rng.standard_normal((2 * B, S * KG)) * 2).astype(np.float32)
    local = (rng.standard_normal((2 * B, S * K, H, W)) * 2).astype(np.float32)
    crit_g = iic.IIDLoss()
    crit_l = iic.IIDSegmentationSmallPathLoss(padding=1, patch_size=1024)

    def step(from_logits):
        tg = torch.from_numpy(glob_rows).to(cuda_device).requires_grad_(True)
        tl = torch.from_numpy(local).to(cuda_device).requires_grad_(True)
        tr = (lambda v: v) if from_logits else (lambda v: (v / T).softmax(1))
        calls = []
        for s in range(S):
            a, b = torch.chunk(tg[:, s * KG:(s + 1) * KG], 2, 0)
            calls.append((crit_g, tr(a), tr(b)))
        for s in range(S):
            a, b = torch.chunk(tl[:, s * K:(s + 1) * K], 2, 0)
            calls.append((crit_l, tr(a), tr(b)))
        out = iic.iic_losses(calls, from_logits=from_logits, T=T)
        sum(o[0] if isinstance(o, tuple) else o for o in out).backward()
        return [float(o[0] if isinstance(o, tuple) else o) for o in out], tg.grad.cpu().numpy(), tl.grad.cpu().numpy()

    names = launched(lambda: step(True))
    assert sum("finish_kernel" in n for n in names) == 1, [n for n in names if "finish" in n]
    assert not any("softmax" in n.lower() for n in names), names
    assert sum("global_backward_kernel<true>" in n for n in names) == S
    f = fused_names(names)
    assert f["stats"] and f["tc"] and f["bwd"]
    vals, gg, gl = step(True)
    vals2, gg2, gl2 = step(False)
    for v, w in zip(vals, vals2):
        assert abs(v - w) <= LOSS_RTOL * max(abs(w), 0.05), (v, w)
    assert relmax(gg, gg2) <= GRAD_RTOL and relmax(gl, gl2) <= GRAD_RTOL
    # oracle: every global term and the first local one
    for s in range(S):
        l1, l2 = glob_rows[:B, s * KG:(s + 1) * KG], glob_rows[B:, s * KG:(s + 1) * KG]
        ol, _, _, og1, og2 = global_oracle(l1, l2, T, 1.0, 1.0, 0.0, None)
        assert abs(vals[s] - ol) <= LOSS_RTOL * max(abs(ol), 0.05)
        assert relmax(gg[:B, s * KG:(s + 1) * KG], og1) <= GRAD_RTOL and relmax(gg[B:, s * KG:(s + 1) * KG], og2) <= GRAD_RTOL
    ol, og1, og2 = oracle(local[:B, :K], local[B:, :K], 1, T)
    assert abs(vals[S] - ol) <= LOSS_RTOL * max(abs(ol), 0.05)
    assert relmax(gl[:B, :K], og1) <= GRAD_RTOL and relmax(gl[B:, :K], og2) <= GRAD_RTOL
