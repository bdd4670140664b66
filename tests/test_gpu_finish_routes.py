"""Every epilogue route of iic_finish at the edges of its rule, and batched terms' gradients, against the fp64 oracle.

iic_finish (csrc/finish.cu) reduces the joints of a whole batch of IIC terms and then runs their epilogues by one of three
routes:

    last-CTA   the last CTA of finish_kernel runs them (option fin_last_cta_epilogue; <= 32 units, <= 1056 doubles)
    batched    batched_epilogue_kernel, one CTA per unit (up to 16384 units)
    per-term   one local_epilogue_kernel / global_epilogue_kernel launch per term (no_fused_epilogue, or > 16384 units)

A unit is one (patch, displacement) of a local term or one global term.  iic_terms (ops.py) also splits a batch into
finish launches of at most 32 terms and sends a global term of more than 4096 rows to the multi-CTA global path.
TERM_SETS puts a batch on each of these thresholds and one step past it, plus the global K at which global_rows_unit
changes its row-group split; test_terms_routing.py restates the rule without a GPU and checks where each set lands.

Every set runs under the default options, fin_last_cta_epilogue and no_fused_epilogue, and asserts from torch.profiler
which finish and epilogue kernels ran.  The maps are one-hot, so every joint is an exact integer count and only the fp64
epilogue separates the kernels from the oracle: each term's float32 loss must lie within 1 ulp of the oracle's loss
rounded to float32 (with the ulp of 0.05 as a floor near 0), each global P must equal the oracle's bit for bit, the
terms of a batch carry different lamda values, and reversing the order of the terms changes no term's bits.

Gradients use random maps, a distinct upstream weight per term and the suite's 1e-4 bound; the batched terms' gradient
routing (test_terms_routing.CASES) runs here with the real kernels against the sum of the oracle's per-use gradients.
"""
import contextlib
import functools
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, relmax

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

GRAD_RTOL = 1e-4
LOSS_FLOOR = 0.05       # below this |loss| the tolerance stays at one float32 ulp of 0.05


def L(B, K, H, W, pad, patch):
    return ("L", B, K, H, W, pad, patch)


def G(N, K):
    return ("G", N, K)


# name = <threshold>_<on | past | value>; test_terms_routing.test_route_rule_places_every_term_set checks each
TERM_SETS = {
    "units32_on": [L(2, 4, 12, 12, 1, 1024)] * 3 + [G(64, 4)] * 5,                      # 27 + 5 units
    "units32_past": [L(2, 4, 12, 12, 1, 1024)] * 3 + [G(64, 4)] * 6,
    "e1056_on": [L(2, 10, 12, 12, 1, 1024), G(64, 12)] + [G(64, 2)] * 3,                # 900 + 144 + 12 doubles
    "e1056_past": [L(2, 10, 12, 12, 1, 1024), G(64, 12), G(64, 3), G(64, 2)],          # 900 + 144 + 9 + 4
    "units16384_on": [L(1, 2, 160, 144, 7, 32), L(1, 2, 96, 80, 1, 32)] + [G(64, 2)] * 4,   # 72*225 + 20*9 + 4
    "units16384_past": [L(1, 2, 160, 144, 7, 32), L(1, 2, 96, 80, 1, 32)] + [G(64, 2)] * 5,
    "terms_32": [L(1, 2, 8, 8, 1, 1024)] * 32,
    "terms_33": [L(1, 2, 8, 8, 1, 1024)] * 33,
    "terms_65": [L(1, 2, 8, 8, 1, 1024)] * 65,
    "rows_4096": [L(2, 4, 12, 12, 1, 1024), G(4096, 4)],
    "rows_4097": [L(2, 4, 12, 12, 1, 1024), G(4097, 4)],
    "globalK_22": [G(300, 22)],
    "globalK_23": [G(300, 23)],
    "globalK_32": [G(300, 32)],
    "globalK_33": [G(300, 33)],
    "globalK_128": [G(300, 128)],
}
OPTS = [{}, {"fin_last_cta_epilogue": 1}, {"no_fused_epilogue": 1}]
OPT_IDS = ["default", "last_cta", "no_fused"]


def lamda_of(i):
    return (1.0, 1.5, 0.5, 2.0)[i % 4]


@pytest.fixture(scope="module")
def iic(cuda_device):
    import iic_b200
    return iic_b200


@contextlib.contextmanager
def options(iic, opts):
    old = {k: iic._lib.set_option(k, v) for k, v in opts.items()}
    try:
        yield
    finally:
        for k, v in old.items():
            iic._lib.set_option(k, v)


def kernels(fn):
    """The set of this library's kernels (bare names) that one call of fn launches."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = {e.name.split("(")[0].split("<")[0].split("::")[-1] for e in prof.events()
             if getattr(e, "device_type", None) is not None and "iic::" in e.name}
    if not names:
        raise RuntimeError("the profiler recorded none of the library's kernels")
    return names


def _finish_side(names):
    return {n for n in names if n == "finish_kernel" or "epilogue" in n}


# ---- one-hot inputs and their oracle results -------------------------------------------------------------------
def _labels(rng, shape, K, block=1):
    """x labels constant over block x block squares of the map, and y labels that agree with them at 70% of the
    positions: every displacement of the window then sees dependent labels, and the loss lies well away from 0."""
    lx = rng.integers(0, K, size=shape)
    if block > 1:
        lx = lx[..., ::block, ::block].repeat(block, -2).repeat(block, -1)
    ly = np.where(rng.random(shape) < 0.7, lx, rng.integers(0, K, size=shape))
    return lx, ly


def _onehot(lab, K, axis):
    return np.moveaxis(np.eye(K, dtype=np.float32)[lab], -1, axis)


@functools.lru_cache(maxsize=None)
def onehot_term(desc, i):
    """float32 (x, y) of term i of a set; the same descriptor and index always give the same maps."""
    rng = np.random.default_rng([i, *desc[1:]])
    if desc[0] == "L":
        _, B, K, H, W, pad, patch = desc
        lx, ly = _labels(rng, (B, H, W), K, 8 if min(H, W) >= 32 else 2)
        return _onehot(lx, K, 1), _onehot(ly, K, 1)
    _, N, K = desc
    lx, ly = _labels(rng, (N,), K)
    return _onehot(lx, K, 1), _onehot(ly, K, 1)


@functools.lru_cache(maxsize=None)
def oracle_term(desc, i):
    """fp64 oracle of term i: the local loss, or the global (loss, loss_no_lamb, P)."""
    x, y = onehot_term(desc, i)
    if desc[0] == "L":
        pad, patch = desc[5], desc[6]
        return O.iid_segmentation_small_path_loss(x, y, pad, (patch, patch), lamda_of(i))
    return O.iid_loss(x, y, lamda_of(i))


def make_batch(iic, name, dev, order):
    """The set's terms in the given order of indices; the terms_* sets are channel blocks of one base tensor."""
    from iic_b200 import ops
    descs = TERM_SETS[name]
    maps = [onehot_term(d, i) for i, d in enumerate(descs)]
    views = {}
    if name.startswith("terms_"):
        B, K, H, W = descs[0][1:5]
        base = torch.from_numpy(np.concatenate([np.concatenate([m[0] for m in maps], 1),
                                                np.concatenate([m[1] for m in maps], 1)], 0)).to(dev).requires_grad_(True)
        for i in range(len(descs)):
            views[i] = (base[:B, i * K:(i + 1) * K], base[B:, i * K:(i + 1) * K])
    else:
        for i, (x, y) in enumerate(maps):
            views[i] = (torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev))
    terms = []
    for i in order:
        d, (x, y) = descs[i], views[i]
        if d[0] == "L":
            p = d[6]
            terms.append(ops.LocalTerm(x, y, None, d[5], (p, p), (p // 2, p // 2), lamda_of(i)))
        else:
            terms.append(ops.GlobalTerm(x, y, lamda_of(i), True))
    return terms


def run_set(iic, name, dev, order):
    """Per term index: the float32 loss (local) or (loss, loss_no_lamb, P) (global), as numpy."""
    from iic_b200 import ops
    out = ops.iic_terms(make_batch(iic, name, dev, order))
    res = {}
    for i, r in zip(order, out):
        res[i] = r.detach().cpu().numpy() if not isinstance(r, tuple) else tuple(v.detach().cpu().numpy() for v in r)
    return res


def f32_close(got, ref):
    """got (float32) within one float32 ulp of ref rounded to float32; the ulp of LOSS_FLOOR near 0."""
    r32 = np.float32(ref)
    tol = np.spacing(np.float32(max(abs(ref), LOSS_FLOOR)))
    return abs(np.float64(got) - np.float64(r32)) <= tol


@pytest.mark.parametrize("opts", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("name", list(TERM_SETS))
def test_route_exact(iic, cuda_device, name, opts):
    import test_terms_routing as R
    descs = TERM_SETS[name]
    fwd = list(range(len(descs)))
    with options(iic, opts):
        got = {}
        names = kernels(lambda: got.update(run_set(iic, name, cuda_device, fwd)))
        rev = run_set(iic, name, cuda_device, fwd[::-1])
    want = R.expected_kernels(descs, opts)
    assert _finish_side(names) == want, (sorted(names), sorted(want))
    for i, d in enumerate(descs):
        ref = oracle_term(d, i)
        if d[0] == "L":
            assert f32_close(got[i], ref), (i, float(got[i]), ref)
            assert got[i].tobytes() == rev[i].tobytes(), (i, float(got[i]), float(rev[i]))
        else:
            assert f32_close(got[i][0], ref[0]) and f32_close(got[i][1], ref[1]), (i, got[i][:2], ref[:2])
            assert np.array_equal(got[i][2], ref[2].astype(np.float32)), (i, np.abs(got[i][2] - ref[2]).max())
            assert all(a.tobytes() == b.tobytes() for a, b in zip(got[i], rev[i])), i


# ---- gradients: random maps, distinct upstream weights ---------------------------------------------------------
def _soft(rng, shape):
    return O.softmax(rng.standard_normal(shape) * 2.0).astype(np.float32)


@pytest.mark.parametrize("opts", OPTS, ids=OPT_IDS)
def test_gradients(iic, cuda_device, opts):
    """A masked term and an unused term on channel blocks of one base, a multi-patch term, a global term whose only used
    output is P and one with both losses used, in one batch small enough for every route."""
    from iic_b200 import ops
    import test_terms_routing as R
    dev = cuda_device
    rng = np.random.default_rng(77)
    B, K, H, W = 2, 4, 16, 16
    u = _soft(rng, (2 * B, 2 * K, H, W))                       # [:, :K] masked term, [:, K:] unused term
    mask = (rng.random((B, 1, H, W)) < 0.8).astype(np.float32)
    mx, my = _soft(rng, (B, 3, 24, 24)), _soft(rng, (B, 3, 24, 24))      # 4 patches of 16 at step 8, padding 0
    gx1, gy1 = _soft(rng, (64, 5)), _soft(rng, (64, 5))
    gx2, gy2 = _soft(rng, (48, 4)), _soft(rng, (48, 4))
    WP = rng.standard_normal((5, 5)).astype(np.float32)
    w = (0.75, 1.25, 3.0, 0.5)

    ud = torch.from_numpy(u).to(dev).requires_grad_(True)
    md = [torch.from_numpy(a).to(dev).requires_grad_(True) for a in (mx, my)]
    gd = [torch.from_numpy(a).to(dev).requires_grad_(True) for a in (gx1, gy1, gx2, gy2)]
    terms = [ops.LocalTerm(ud[:B, :K], ud[B:, :K], torch.from_numpy(mask).to(dev), 1, (H, W), (H, W), 1.5),
             ops.LocalTerm(md[0], md[1], None, 0, (16, 16), (8, 8), 0.5),
             ops.LocalTerm(ud[:B, K:], ud[B:, K:], None, 1, (H, W), (H, W), 1.0),
             ops.GlobalTerm(gd[0], gd[1], 2.0, True),
             ops.GlobalTerm(gd[2], gd[3], 1.0, True)]
    with options(iic, opts):
        out = ops.iic_terms(terms)
        tot = w[0] * out[0] + w[1] * out[1] + (out[3][2] * torch.from_numpy(WP).to(dev)).sum() \
            + w[2] * out[4][0] + w[3] * out[4][1]
        with R.poisoned_empty():
            tot.backward()
    g = ud.grad.cpu().numpy()
    _, ogx, ogy = O.iid_segmentation_small_path_loss(u[:B, :K], u[B:, :K], 1, (H, W), 1.5, mask=mask, with_grads=True)
    assert relmax(g[:B, :K], w[0] * ogx) <= GRAD_RTOL and relmax(g[B:, :K], w[0] * ogy) <= GRAD_RTOL
    assert not g[:, K:].any(), "the unused term's blocks must hold exact zeros"
    _, ogx, ogy = O.iid_segmentation_small_path_loss(mx, my, 0, (16, 16), 0.5, with_grads=True)
    assert relmax(md[0].grad.cpu().numpy(), w[1] * ogx) <= GRAD_RTOL
    assert relmax(md[1].grad.cpu().numpy(), w[1] * ogy) <= GRAD_RTOL
    ox, oy = O.iid_loss_grads(gx1, gy1, 2.0, g_loss=0.0, g_loss_no_lamb=0.0, g_P=WP)
    assert relmax(gd[0].grad.cpu().numpy(), ox) <= GRAD_RTOL and relmax(gd[1].grad.cpu().numpy(), oy) <= GRAD_RTOL
    ox, oy = O.iid_loss_grads(gx2, gy2, 1.0, g_loss=w[2], g_loss_no_lamb=w[3])
    assert relmax(gd[2].grad.cpu().numpy(), ox) <= GRAD_RTOL and relmax(gd[3].grad.cpu().numpy(), oy) <= GRAD_RTOL


# ---- the routing matrix of test_terms_routing with the real kernels -----------------------------------------------
def _oracle_use_grads(kind, x, y, use, term):
    """fp64 oracle gradients (gx, gy) of one term's used outputs, weighted as test_terms_routing.objective weights
    them; x, y float64 numpy."""
    import test_terms_routing as R
    if kind == "G":
        w1, w2, w3 = use
        K = x.shape[1]
        return O.iid_loss_grads(x, y, term.lamb, g_loss=w1 or 0.0, g_loss_no_lamb=w2 or 0.0,
                                g_P=None if w3 is None else w3 * R.p_weights(K, torch.zeros(())).double().numpy())
    _, gx, gy = O.iid_segmentation_small_path_loss(x, y, term.pad, term.patch, term.lamda, with_grads=True)
    return use * gx, use * gy


@pytest.mark.parametrize("side", [False, True], ids=["main_stream", "side_stream"])
def test_routing_end_to_end(iic, cuda_device, monkeypatch, side):
    import test_terms_routing as R
    from iic_b200 import ops
    monkeypatch.setattr(ops, "overlap_global_backward", side)
    rng = np.random.default_rng(5)
    for name, shape, build in R.CASES:
        init = torch.from_numpy(O.softmax(rng.standard_normal(shape), axis=1)).float()
        base = init.to(cuda_device).requires_grad_(True)
        spec, terms = R.make_terms(build, base)
        outs = ops.iic_terms(terms)
        with R.poisoned_empty():
            R.objective(spec, outs).backward()
        ref = init.double().requires_grad_(True)
        spec_r, terms_r = R.make_terms(build, ref)
        tot = 0
        for (kind, x, y, use), t in zip(spec_r, terms_r):
            if use is None or (kind == "G" and all(u_ is None for u_ in use)):
                continue
            gx, gy = _oracle_use_grads(kind, x.detach().numpy(), y.detach().numpy(), use, t)
            tot = tot + (x * torch.from_numpy(gx)).sum() + (y * torch.from_numpy(gy)).sum()
        tot.backward()
        got, want = base.grad.cpu().numpy(), ref.grad.numpy()
        assert relmax(got, want) <= GRAD_RTOL, (name, relmax(got, want))
        assert not got[want == 0].any(), (name, "elements no used term reads must get exact zeros")


def test_simplex_check_in_second_chunk(iic, cuda_device):
    """Strict mode: a non-simplex term placed in the second finish launch of a 40-term batch still raises."""
    dev = cuda_device
    rng = np.random.default_rng(3)
    crit = iic.IIDSegmentationLoss(padding=1)

    def calls(bad):
        out = []
        for i in range(40):
            x, y = _soft(rng, (1, 2, 8, 8)), _soft(rng, (1, 2, 8, 8))
            if i == bad:
                x = x * 1.5
            out.append((crit, torch.from_numpy(x).to(dev).requires_grad_(True),
                        torch.from_numpy(y).to(dev).requires_grad_(True)))
        return out
    with iic.checks.check_mode("strict"):
        iic.iic_losses(calls(None))
        with pytest.raises(AssertionError):
            iic.iic_losses(calls(35))
        iic.iic_losses(calls(None))          # the flag was cleared with the raise
