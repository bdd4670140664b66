"""The cluster head's softmax fused into the local IIC term for 16 <= K <= 24 (the reference's config uses 20 clusters,
paddings 1 and 3): the per-pixel softmax statistics pass, the from-logits packed tensor-core joint and the from-logits
row-block tensor-core backward, reached through IIDSegmentationSmallPathLoss.from_logits and iic_losses(from_logits=True).

Losses and LOGIT gradients are compared with the fp64 oracle chained through its own softmax (O.softmax,
O.softmax_backward with T) at the project's bounds: loss 1e-5 relative, gradients 1e-4 max-norm relative.  Which
kernels ran is read from torch.profiler (full names, so that the from-logits instantiations <T, true> are told apart)."""
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
    base = rng.standard_normal((B, K, max(H // 4, 1), max(W // 4, 1))).repeat(4, axis=2).repeat(4, axis=3)[:, :, :H, :W] * 3
    if base.shape[2] < H or base.shape[3] < W:
        base = np.pad(base, ((0, 0), (0, 0), (0, H - base.shape[2]), (0, W - base.shape[3])), mode="edge")
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
            "tcp": any("local_joint_tcp_kernel<" in n and "true>" in n for n in names),
            "tcrb": any("local_bwd_tcrb_kernel<" in n and "true>" in n for n in names),
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
    print(f"loss rel {abs(loss - ol) / abs(ol):.2e}  grad relmax {max(ex, ey):.2e}")
    assert ex <= GRAD_RTOL and ey <= GRAD_RTOL, (ex, ey)


# ---------------------------------------------------------------------------------------------------
# against the oracle: K x padding x temperature, correlated and sharply peaked logits
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("peaked", [False, True])
@pytest.mark.parametrize("T", [1.0, 0.1])
@pytest.mark.parametrize("pad", [1, 3])
@pytest.mark.parametrize("K", [16, 20, 24])
def test_from_logits_vs_oracle(iic, cuda_device, K, pad, T, peaked):
    rng = np.random.default_rng(1000 * K + 10 * pad + int(10 * T) + peaked)
    B, H, W = 2, 40, 64
    # peaked: logits scaled so that l / T spans hundreds (T = 0.1: several hundred), p one-hot up to fp32
    l1, l2 = logit_views(rng, B, K, H, W, scale=8.0 if peaked else 1.0)
    with options(iic, tcrb_p1=1):                 # padding 1 at a small map: past the "fill the SMs" gate
        a = torch.from_numpy(l1).to(cuda_device)
        assert iic.ops.from_logits_covered(a, a, pad)
        loss, ga, gb = run_from_logits(iic, cuda_device, l1, l2, pad, T)
    check(loss, ga, gb, *oracle(l1, l2, pad, T, 0.37))


# ---------------------------------------------------------------------------------------------------
# the kernels' edges: B = 1, H not a multiple of the row block, the backward's column panels, border pixels
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,K,H,W,pad", [
    (1, 20, 24, 64, 3),       # B = 1
    (2, 20, 23, 128, 3),      # W = 128: one panel, one 128-pixel tile; R = 21 does not divide H = 23
    (2, 20, 13, 144, 1),      # W = 144: one panel, two tiles (R = 10)
    (1, 20, 12, 256, 3),      # W = 256: two 128-column panels
    (1, 20, 11, 272, 1),      # W = 272: two 136-column panels
    (2, 20, 16, 32, 3),       # 7 x 7 window on a 16 x 32 map: most joint terms touch the zero padding
    (3, 17, 16, 32, 3),       # odd K: channels 17..23 of the staged boxes must stay zero
])
def test_from_logits_edges(iic, cuda_device, B, K, H, W, pad):
    rng = np.random.default_rng(B * 7 + K * 11 + H * 13 + W + pad)
    l1, l2 = logit_views(rng, B, K, H, W)
    with options(iic, tcrb_p1=1):
        names = launched(lambda: run_from_logits(iic, cuda_device, l1, l2, pad, 0.5))
        loss, ga, gb = run_from_logits(iic, cuda_device, l1, l2, pad, 0.5)
    f = fused_names(names)
    assert f["stats"] and f["tcp"] and f["tcrb"] and not f["softmax"], names
    check(loss, ga, gb, *oracle(l1, l2, pad, 0.5, 0.37))


def test_from_logits_repeatable(iic, cuda_device):
    """Two identical calls give bit-identical loss and gradients."""
    rng = np.random.default_rng(3)
    l1, l2 = logit_views(rng, 2, 20, 40, 144)
    with options(iic, tcrb_p1=1):
        r1 = run_from_logits(iic, cuda_device, l1, l2, 1, 0.1)
        r2 = run_from_logits(iic, cuda_device, l1, l2, 1, 0.1)
    r3 = run_from_logits(iic, cuda_device, l1, l2, 3, 1.0)
    r4 = run_from_logits(iic, cuda_device, l1, l2, 3, 1.0)
    for u, v in ((r1, r2), (r3, r4)):
        assert u[0] == v[0]
        assert np.array_equal(u[1], v[1]) and np.array_equal(u[2], v[2])


# ---------------------------------------------------------------------------------------------------
# channel blocks of one (2B, S*K, H, W) head output: gradients land in their blocks, nothing else is written
# ---------------------------------------------------------------------------------------------------
def test_blocks_of_head_output_and_sentinels(iic, cuda_device):
    S, B, K, H, W, pad, T = 5, 2, 20, 24, 64, 3, 0.5
    rng = np.random.default_rng(11)
    full = rng.standard_normal((2 * B, S * K, H, W)).astype(np.float32) * 2
    t = torch.from_numpy(full).to(cuda_device).requires_grad_(True)
    halves = torch.chunk(t, 2, 0)                                     # the epocher's (view 1, view 2) split
    crit = iic.IIDSegmentationSmallPathLoss(padding=pad, patch_size=4096)
    for s in (1, 3):
        a, b = halves[0][:, s * K:(s + 1) * K], halves[1][:, s * K:(s + 1) * K]
        loss = crit.from_logits(a, b, T=T)
        loss.backward()
    g = t.grad.cpu().numpy()
    for s in range(S):
        blk = g[:, s * K:(s + 1) * K]
        if s in (1, 3):
            l1, l2 = full[:B, s * K:(s + 1) * K], full[B:, s * K:(s + 1) * K]
            _, og1, og2 = oracle(l1, l2, pad, T)
            assert relmax(blk[:B], og1) <= GRAD_RTOL and relmax(blk[B:], og2) <= GRAD_RTOL
        else:
            assert not blk.any()

    # the raw backward entry point writing into channel-block views of sentinel-filled tensors
    lx = torch.from_numpy(full[:B]).to(cuda_device).contiguous()
    ly = torch.from_numpy(full[B:]).to(cuda_device).contiguous()
    a, b = lx[:, 2 * K:3 * K], ly[:, 2 * K:3 * K]
    term = iic.ops.LocalTerm(a, b, None, pad, (H, W), (H, W), 1.0, logits=True, inv_temperature=1.0 / T)
    (r,) = iic.ops._finish_terms([term], False)
    assert r["stats"] is not None
    GX = torch.full((B, S * K, H, W), 7.25, device=cuda_device)
    GY = torch.full((B, S * K, H, W), -3.5, device=cuda_device)
    gx, gy = GX[:, 2 * K:3 * K], GY[:, 2 * K:3 * K]
    gx.fill_(float("nan"))
    gy.fill_(float("nan"))
    iic.ops._local_backward_logits_stats_into(a, b, r["stats"], r["Wx"], r["Wy"], torch.ones((), device=cuda_device), pad,
                                             1.0 / T, gx, gy)
    _, og1, og2 = oracle(full[:B, 2 * K:3 * K], full[B:, 2 * K:3 * K], pad, T)
    assert relmax(gx.cpu().numpy(), og1) <= GRAD_RTOL and relmax(gy.cpu().numpy(), og2) <= GRAD_RTOL
    GX[:, 2 * K:3 * K] = 7.25
    GY[:, 2 * K:3 * K] = -3.5
    assert bool((GX == 7.25).all()) and bool((GY == -3.5).all())


# ---------------------------------------------------------------------------------------------------
# dispatch: covered shapes run the fused kernels and no torch softmax; the query agrees with what ran
# ---------------------------------------------------------------------------------------------------
def sms(iic):
    return iic._lib.load().iic_b200_sm_count(0)


@pytest.mark.parametrize("B,K,H,W,pad,opts,fused", [
    (4, 20, 32, 64, 3, {}, True),                        # padding 3
    (32, 20, 224, 224, 1, {}, True),                     # padding 1 with enough row blocks
    (2, 20, 32, 72, 3, {}, False),                       # W % 16 != 0
    (2, 20, 32, 64, 2, {}, False),                       # padding 2
    (4, 20, 32, 64, 3, {"no_tc": 1}, False),             # tensor cores switched off
    (4, 20, 32, 64, 3, {"no_tma": 1}, False),            # TMA switched off
    (8, 20, 112, 112, 1, {}, None),                      # config 3 Up_conv3: the padding-1 gate decides
    (2, 20, 32, 64, 1, {}, False),                       # padding 1 below the gate
    (2, 20, 32, 64, 1, {"tcrb_p1": 1}, True),            # ... unless forced
    (2, 12, 32, 64, 3, {}, False),                       # K outside 16..24
])
def test_query_matches_what_ran(iic, cuda_device, B, K, H, W, pad, opts, fused):
    rng = np.random.default_rng(B + K + H + W + pad)
    l1, l2 = logit_views(rng, B, K, H, W)
    with options(iic, **opts):
        a = torch.from_numpy(l1).to(cuda_device)
        b = torch.from_numpy(l2).to(cuda_device)
        covered = iic.ops.from_logits_covered(a, b, pad)
        if fused is None:        # (8, 20, 112, 112): 8 * ceil(112 / 21) = 48 row blocks
            fused = 8 * -(-112 // 21) >= 2 * sms(iic)
        assert covered == fused
        names = launched(lambda: run_from_logits(iic, cuda_device, l1, l2, pad, 1.0))
    f = fused_names(names)
    if fused:
        assert f["stats"] and f["tcp"] and f["tcrb"] and not f["softmax"], names
    else:
        assert not (f["stats"] or f["tcp"] or f["tcrb"]) and f["softmax"], names
    print(f"{(B, K, H, W, pad, opts)}: {'fused' if fused else 'softmax + probability path'}")


# ---------------------------------------------------------------------------------------------------
# the batched API from logits: a config-3-like iteration in ONE finish launch
# ---------------------------------------------------------------------------------------------------
def test_iic_losses_from_logits_config3(iic, cuda_device):
    """5 sub-heads x {global, padding 1, padding 3} from logits, plus one uncovered term (W % 16 != 0), against
    iic_losses on the softmaxed maps and against the oracle; the whole batch runs one finish launch."""
    S, B, K, T = 5, 2, 20, 0.5
    rng = np.random.default_rng(2026)
    g_l = [(rng.standard_normal((B, K)) * 2).astype(np.float32) for _ in range(2 * S)]
    heads = {}
    for name, (H, W) in {"p1": (16, 32), "p3": (32, 48), "odd": (16, 40)}.items():
        heads[name] = (rng.standard_normal((2 * B, S * K, H, W)) * 2).astype(np.float32)
    glob = iic.IIDLoss()
    c1 = iic.IIDSegmentationSmallPathLoss(padding=1, patch_size=1024)
    c3 = iic.IIDSegmentationSmallPathLoss(padding=3, patch_size=1024)

    def calls(transform):
        tg = [torch.from_numpy(a).to(cuda_device).requires_grad_(True) for a in g_l]
        th = {k: torch.from_numpy(v).to(cuda_device).requires_grad_(True) for k, v in heads.items()}
        cs = []
        for s in range(S):
            cs.append((glob, transform(tg[2 * s]), transform(tg[2 * s + 1])))
        for name, crit in (("p1", c1), ("p3", c3), ("odd", c3)):
            h = th[name].view(2 * B, S, K, *th[name].shape[2:])
            for s in range(S if name != "odd" else 1):
                a, b = torch.chunk(h[:, s], 2, 0)
                cs.append((crit, transform(a), transform(b)))
        return tg, th, cs

    with options(iic, tcrb_p1=1):
        tg, th, cs = calls(lambda v: v)
        assert [iic.ops.from_logits_covered(c[1], c[2], c[0].padding) for c in cs[S:]] == [True] * (2 * S) + [False]
        names = []

        def fused_step():
            out = iic.iic_losses(cs, from_logits=True, T=T)
            tot = sum(o[0] if isinstance(o, tuple) else o for o in out)
            tot.backward()
            return out
        names = launched(fused_step)
        assert sum("finish_kernel" in n for n in names) == 1, [n for n in names if "finish" in n]
        for g in tg:
            g.grad = None
        for h in th.values():
            h.grad = None
        out = fused_step()
        grads = [g.grad.cpu().numpy() for g in tg] + [h.grad.cpu().numpy() for h in th.values()]

        tg2, th2, cs2 = calls(lambda v: (v / T).softmax(1))
        out2 = iic.iic_losses(cs2)
        sum(o[0] if isinstance(o, tuple) else o for o in out2).backward()
        grads2 = [g.grad.cpu().numpy() for g in tg2] + [h.grad.cpu().numpy() for h in th2.values()]

    vals = [float(o[0] if isinstance(o, tuple) else o) for o in out]
    vals2 = [float(o[0] if isinstance(o, tuple) else o) for o in out2]
    # padding 1 runs different joints on the two sides (tcp from logits vs FFMA2 on probabilities): the project's bounds
    for v, w in zip(vals, vals2):
        assert abs(v - w) <= LOSS_RTOL * max(abs(w), 0.05), (v, w)
    for g, h in zip(grads, grads2):
        assert relmax(g, h) <= GRAD_RTOL

    # oracle: the local terms and the first global term
    k = S
    for name, pad in (("p1", 1), ("p3", 3), ("odd", 3)):
        hv = heads[name].reshape(2 * B, S, K, *heads[name].shape[2:])
        gh = grads[2 * S + list(heads).index(name)].reshape(hv.shape)
        for s in range(S if name != "odd" else 1):
            ol, og1, og2 = oracle(hv[:B, s], hv[B:, s], pad, T)
            assert abs(vals[k] - ol) <= LOSS_RTOL * max(abs(ol), 0.05), (name, s, vals[k], ol)
            assert relmax(gh[:B, s], og1) <= GRAD_RTOL and relmax(gh[B:, s], og2) <= GRAD_RTOL
            k += 1
    p1, p2 = O.softmax(g_l[0], 1, T), O.softmax(g_l[1], 1, T)
    o1 = O.iid_loss(p1, p2)[0]
    ox, oy = O.iid_loss_grads(p1, p2)
    assert abs(vals[0] - o1) <= LOSS_RTOL * max(abs(o1), 0.05)
    assert relmax(grads[0], O.softmax_backward(p1, ox, 1, T)) <= GRAD_RTOL


def test_iic_losses_from_logits_refuses_masks(iic, cuda_device):
    a = torch.zeros(1, 20, 16, 32, device=cuda_device, requires_grad=True)
    b = torch.zeros(1, 20, 16, 32, device=cuda_device, requires_grad=True)
    m = torch.ones(1, 1, 16, 32, device=cuda_device)
    with pytest.raises(ValueError):
        iic.iic_losses([(iic.IIDSegmentationSmallPathLoss(padding=3, patch_size=1024), a, b, m)], from_logits=True)
