"""Gradient routing of batched IIC terms (ops.IICTermsFunction), and where each batch's epilogues run.

iic_terms hands every term's x / y to IICTermsFunction as (source, block) pairs: the distinct differentiable tensors
behind the views and, for a channel block of a contiguous tensor, its (n0, c0) offset.  The backward then writes each
term's gradient straight into its block of the source's gradient buffer, zero-fills only the sources that need it, adds
a second use of a block through a temporary, and can run the global terms' gradients on a side stream.  A misrouted,
dropped or overwritten write is invisible in the loss and shows up only in a gradient.

The routing matrix below checks it on the CPU with the kernels replaced by stubs: every use's gradient is a constant
distinct per term and per x / y (1 + term and 100 + term for a local term, more for a global term's three outputs) times
the upstream gradient, and the result must EQUAL what autograd gives for the same linear functional over the same views.
The constants and weights are small integers, so every sum is exact.  torch.empty hands out NaN-filled tensors inside
the backward, so an element that no use writes shows up too.

The second half restates iic_finish's choice of epilogue route (csrc/finish.cu) and iic_terms' batch splits in Python,
and checks that each term set of test_gpu_finish_routes.py lands where its name says.
"""
import contextlib
import os
import sys

import pytest
import torch

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_oracle as O  # noqa: E402

import iic_b200  # noqa: E402,F401
from iic_b200 import ops  # noqa: E402

GLOBAL_K = 4          # column width of the global blocks of the 2-D bases below


# ---- the routing matrix: (name, base shape, build) with build(base) -> [(kind, x, y, use), ...] --------------------
# kind "L": local term on 4-D views, use = upstream weight of its loss or None (unused); "Lp": the same with several
# patches (the kernels accumulate into their output); "G": global term on 2-D views, use = weights of
# (loss, loss_no_lamb, P), each None when that output is unused.
def _heads(t, S, K, w=1):
    B = t.shape[0] // 2
    return [("L", t[:B, s * K:(s + 1) * K], t[B:, s * K:(s + 1) * K], w + s % 3) for s in range(S)]


CASES = [
    ("disjoint_chunks", (4, 20, 8, 8),
     lambda t: [("L", *torch.chunk(t[:, :10], 2, 0), 1), ("L", *torch.chunk(t[:, 10:], 2, 0), 2)]),
    ("same_block_as_x_and_y", (4, 20, 8, 8), lambda t: [("L", t[:2, :10], t[:2, :10], 1)]),
    ("same_block_in_two_terms", (4, 20, 8, 8),
     lambda t: [("L", t[:2, :10], t[2:, :10], 1), ("L", t[:2, :10], t[2:, 10:], 2)]),
    ("forty_terms_two_chunks", (4, 40, 8, 8),
     lambda t: [("L", t[:2, k:k + 2], t[2:, k:k + 2], 1 + k % 3) for k in range(0, 40, 2)] * 2),
    ("blocks_not_tiling", (4, 20, 8, 8), lambda t: [("L", t[:1, 3:7], t[2:3, 3:7], 1)]),
    ("overlapping_channel_blocks", (4, 20, 8, 8), lambda t: [("L", t[:2, 0:10], t[:2, 5:15], 1)]),
    ("overlapping_blocks_sum_to_numel", (4, 10, 8, 8), lambda t: [("L", t[0:2], t[1:3], 1)]),
    ("whole_leaf_and_its_blocks", (4, 10, 8, 8), lambda t: [("L", t, t, 1), ("L", t[:2], t[2:], 2)]),
    ("whole_nonleaf_and_its_blocks", (4, 10, 8, 8),
     lambda t: (lambda m: [("L", m, m, 1), ("L", m[:2], m[2:], 2)])(t * 1)),
    ("global_blocks_2d", (6, 3 * GLOBAL_K),
     lambda t: [("G", t[:3, s * GLOBAL_K:(s + 1) * GLOBAL_K], t[3:, s * GLOBAL_K:(s + 1) * GLOBAL_K], (1 + s, 2, 1))
                for s in range(3)]),
    ("global_overlapping_2d", (6, 3 * GLOBAL_K),
     lambda t: [("G", t[:3, 0:GLOBAL_K], t[3:, 0:GLOBAL_K], (1, 1, None)),
                ("G", t[:3, 2:2 + GLOBAL_K], t[2:5, 2:2 + GLOBAL_K], (2, None, None))]),
    ("unused_term", (4, 20, 8, 8),
     lambda t: [("L", t[:2, :10], t[2:, :10], None), ("L", t[:2, 10:], t[2:, 10:], 1)]),
    ("global_P_only", (6, 2 * GLOBAL_K),
     lambda t: [("G", t[:3, :GLOBAL_K], t[3:, :GLOBAL_K], (None, None, 1)),
                ("G", t[:3, GLOBAL_K:], t[3:, GLOBAL_K:], (2, None, None))]),
    ("local_and_global_one_base", (4, 20, 8, 8),
     lambda t: [("L", t[:2, :10], t[2:, :10], 1),
                ("G", t.view(4, -1)[:, 700:700 + GLOBAL_K], t.view(4, -1)[:, 1200:1200 + GLOBAL_K], (1, 1, None))]),
    ("local_and_global_overlapping", (4, 20, 8, 8),
     lambda t: [("L", t[:2, :10], t[2:, :10], 1),
                ("G", t.view(4, -1)[:, 60:60 + GLOBAL_K], t.view(4, -1)[:, 700:700 + GLOBAL_K], (1, None, 2))]),
    ("multi_patch_blocks", (4, 20, 8, 8),
     lambda t: [("Lp", t[:2, :10], t[2:, :10], 1), ("Lp", t[:2, 5:15], t[2:, 10:], 2)]),
    ("33_terms_one_base", (4, 33 * 2, 4, 4), lambda t: _heads(t, 33, 2)),
    ("65_terms_one_base", (4, 65 * 2, 4, 4), lambda t: _heads(t, 65, 2)),
]
LOCAL_C = (1, 100)                        # per-use constants: + term index
GLOBAL_C = ((1, 100), (1000, 2000), (3000, 4000))     # (x, y) per output: loss, loss_no_lamb, P


def make_terms(build, base):
    """LocalTerm / GlobalTerm objects (padding 1; one patch, or four for "Lp") and their uses."""
    spec = build(base)
    terms = []
    for kind, x, y, use in spec:
        if kind == "G":
            terms.append(ops.GlobalTerm(x, y, 1.0, True))
        else:
            H, W = x.shape[2:]
            p = (H // 2, W // 2) if kind == "Lp" else (H, W)
            terms.append(ops.LocalTerm(x, y, None, 1, p, (p[0] // 2, p[1] // 2) if kind == "Lp" else p, 1.0))
    return spec, terms


def p_weights(K, like):
    """The upstream gradient of P per unit weight: 1, 2, ..., K*K (a uniform one would be orthogonal to P, whose
    entries sum to 1)."""
    return torch.arange(1, K * K + 1, dtype=like.dtype, device=like.device).view(K, K)


def objective(spec, outs):
    """sum over the used outputs of weight * output (P enters as weight * (p_weights * P).sum())."""
    tot = 0
    for (kind, x, y, use), o in zip(spec, outs):
        if kind == "G":
            for w, v in zip(use, (o[0], o[1], (p_weights(o[2].shape[0], o[2]) * o[2]).sum())):
                if w is not None:
                    tot = tot + w * v
        elif use is not None:
            tot = tot + use * o
    return tot


def reference_outputs(spec):
    """Per term the outputs of plain tensor expressions whose gradients are the stubs' constants."""
    outs = []
    for i, (kind, x, y, use) in enumerate(spec):
        if kind == "G":
            lin = [(cx + i) * x.sum() + (cy + i) * y.sum() for cx, cy in GLOBAL_C]
            K = x.shape[1]
            outs.append((lin[0], lin[1], lin[2] * torch.ones(K, K)))
        else:
            outs.append((LOCAL_C[0] + i) * x.sum() + (LOCAL_C[1] + i) * y.sum())
    return outs


class _Stream:
    def wait_stream(self, other):
        pass


@pytest.fixture
def stubbed(monkeypatch):
    """Kernels replaced by the constant stubs; the CUDA stream calls of the side-stream branch by no-ops.  The test
    fills the returned dict with id(term) -> the term's index in its whole list (a batch may be split)."""
    index = {}

    def fake_finish(terms, check_simplex):
        recs = []
        for t in terms:
            i = index[id(t)]
            x, y = t.x.detach(), t.y.detach()
            if isinstance(t, ops.LocalTerm):
                H, W = x.shape[2:]
                npatch = len(O.patch_windows(H, W, t.patch, t.step))
                recs.append(dict(kind="local", x=x, y=y, mask=None, Wx=torch.full((1,), float(i)), Wy=torch.zeros(1),
                                 loss=torch.zeros(()), K=x.shape[1], T=3, npatch=npatch, joff=0, E=1))
            else:
                K = x.shape[1]
                recs.append(dict(kind="global", x=x, y=y, P=torch.zeros(K, K), loss=torch.zeros(()),
                                 loss_nl=torch.zeros(()), J=torch.full((K * K,), float(i), dtype=torch.float64), K=K,
                                 joff=0, E=K * K))
        return recs

    def fake_local(x, y, mask, Wx, Wy, g, pad, ph, pw, sh, sw, gx, gy):
        i = int(Wx[0])
        multi = (ph, pw) != tuple(x.shape[2:])
        for dst, c in ((gx, LOCAL_C[0] + i), (gy, LOCAL_C[1] + i)):
            if multi:                            # the multi-patch kernels accumulate into their output
                dst.add_(c * g)
            else:
                dst.copy_((c * g).expand_as(dst))

    def fake_global(x, y, J, lamb, symmetric, g1, g2, gP, gx, gy):
        i = int(J.view(-1)[0])
        for dst, col in ((gx, 0), (gy, 1)):
            v = torch.zeros(())
            for g, c in zip((g1, g2, None if gP is None else gP.sum()), GLOBAL_C):
                if g is not None:
                    v = v + (c[col] + i) * g
            dst.copy_(v.expand_as(dst))

    monkeypatch.setattr(ops, "_finish_terms", fake_finish)
    monkeypatch.setattr(ops, "_local_backward_into", fake_local)
    monkeypatch.setattr(ops, "_global_backward_into", fake_global)
    monkeypatch.setattr(ops, "_side_stream", lambda dev: _Stream())
    monkeypatch.setattr(torch.cuda, "current_stream", lambda dev=None: _Stream())
    monkeypatch.setattr(torch.cuda, "stream", lambda s: contextlib.nullcontext())
    return index


@contextlib.contextmanager
def poisoned_empty():
    """torch.empty returns NaN-filled floating tensors: memory nobody writes cannot pass for zeros."""
    real = torch.empty

    def empty(*a, **k):
        t = real(*a, **k)
        return t.fill_(float("nan")) if t.is_floating_point() else t
    torch.empty = empty
    try:
        yield
    finally:
        torch.empty = real


@pytest.fixture(params=[False, True], ids=["main_stream", "side_stream"])
def overlap_flag(request, monkeypatch):
    monkeypatch.setattr(ops, "overlap_global_backward", request.param)
    return request.param


@pytest.mark.parametrize("name,shape,build", CASES, ids=[c[0] for c in CASES])
def test_routing_matrix(stubbed, overlap_flag, name, shape, build):
    base = torch.zeros(shape, requires_grad=True)
    spec, terms = make_terms(build, base)
    stubbed.update({id(t): i for i, t in enumerate(terms)})
    outs = ops.iic_terms(terms)
    with poisoned_empty():
        objective(spec, outs).backward()
    ref = torch.zeros(shape, requires_grad=True)
    spec_r, _ = make_terms(build, ref)
    objective(spec_r, reference_outputs(spec_r)).backward()
    assert base.grad is not None and ref.grad is not None
    bad = (base.grad != ref.grad).nonzero()
    assert torch.equal(base.grad, ref.grad), (name, bad[:8].tolist(), base.grad[tuple(bad[0])].item() if len(bad) else None)


def test_disjoint_tiling_blocks_skip_the_zero_fill(stubbed):
    """Disjoint blocks that tile their source are written in place into a torch.empty buffer: no zero fill, no
    temporaries (the config-3 sub-head layout)."""
    base = torch.zeros((4, 20, 8, 8), requires_grad=True)
    spec, terms = make_terms(lambda t: _heads(t, 10, 2), base)
    stubbed.update({id(t): i for i, t in enumerate(terms)})
    outs = ops.iic_terms(terms)
    calls = []
    real_zeros, real_zeros_like = torch.zeros, torch.zeros_like
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(torch, "zeros", lambda *a, **k: calls.append("zeros") or real_zeros(*a, **k))
        mp.setattr(torch, "zeros_like", lambda *a, **k: calls.append("zeros_like") or real_zeros_like(*a, **k))
        with poisoned_empty():
            objective(spec, outs).backward()
    assert calls == [] and not base.grad.isnan().any()


# ---- iic_finish's epilogue route and iic_terms' splits, restated ---------------------------------------------------
FIN_SMALL_UNITS = 32          # csrc/finish.cu
FIN_MAX_PATCHES = 256
FIN_STAGE_DOUBLES = 32 * 33   # FIN_WARPS * 33
FIN_BIG_MAX_UNITS = 16384


def n_patches(t):
    """t = ("L", B, K, H, W, pad, patch[, ...]) -> patch windows (step = patch // 2); 1 for a global term."""
    if t[0] != "L":
        return 1
    H, W, patch = t[3], t[4], t[6]
    return len(O.patch_windows(H, W, (patch, patch), (patch // 2, patch // 2)))


def term_units(t):
    """Epilogue units (one per (patch, displacement), one per global term) and joint doubles E of one term."""
    if t[0] == "L":
        T = 2 * t[5] + 1
        return n_patches(t) * T * T, n_patches(t) * T * T * t[2] * t[2]
    return 1, t[2] * t[2]


def finish_route(terms, opts):
    """csrc/finish.cu iic_finish: which kernels run the epilogues of one finish launch."""
    units = sum(term_units(t)[0] for t in terms)
    E = sum(term_units(t)[1] for t in terms)
    patches = sum(n_patches(t) for t in terms if t[0] == "L")
    fused = not opts.get("no_fused_epilogue")
    small = fused and units <= FIN_SMALL_UNITS and patches <= FIN_MAX_PATCHES and E <= FIN_STAGE_DOUBLES
    if small and opts.get("fin_last_cta_epilogue"):
        return "last_cta"
    if fused and units <= FIN_BIG_MAX_UNITS:
        return "batched"
    return "per_term"


def split(terms):
    """ops.iic_terms: global terms of more than GLOBAL_ROWS_MAX rows leave the batch; the rest go to finish launches
    of at most MAX_TERMS_PER_FINISH terms.  Returns (finish batches, split-off global terms)."""
    alone = [t for t in terms if t[0] == "G" and t[1] > ops.GLOBAL_ROWS_MAX]
    rest = [t for t in terms if not (t[0] == "G" and t[1] > ops.GLOBAL_ROWS_MAX)]
    step = ops.MAX_TERMS_PER_FINISH
    return [rest[i:i + step] for i in range(0, len(rest), step)], alone


ROUTE_KERNELS = {"last_cta": {"finish_kernel"}, "batched": {"finish_kernel", "batched_epilogue_kernel"}}


def expected_kernels(terms, opts):
    """The finish and epilogue kernels that one evaluation of `terms` launches."""
    batches, alone = split(terms)
    out = set()
    for b in batches:
        r = finish_route(b, opts)
        if r == "per_term":
            out |= {"finish_kernel"} | {"local_epilogue_kernel" if t[0] == "L" else "global_epilogue_kernel" for t in b}
        else:
            out |= ROUTE_KERNELS[r]
    if alone:
        out.add("global_epilogue_kernel")
    return out


def test_route_rule_places_every_term_set():
    """Each term set of the GPU module sits where its name says: on a threshold or one step past it."""
    import test_gpu_finish_routes as G
    seen = set()
    for name, terms in G.TERM_SETS.items():
        units = sum(term_units(t)[0] for t in terms)
        E = sum(term_units(t)[1] for t in terms)
        batches, alone = split(terms)
        thr, side = name.rsplit("_", 1)
        seen.add(thr)
        if thr == "units32":
            assert units == {"on": 32, "past": 33}[side] and E <= FIN_STAGE_DOUBLES
            assert finish_route(terms, {"fin_last_cta_epilogue": 1}) == {"on": "last_cta", "past": "batched"}[side]
        elif thr == "e1056":
            assert E == {"on": 1056, "past": 1057}[side] and units <= FIN_SMALL_UNITS
            assert finish_route(terms, {"fin_last_cta_epilogue": 1}) == {"on": "last_cta", "past": "batched"}[side]
        elif thr == "units16384":
            assert units == {"on": 16384, "past": 16385}[side]
            assert finish_route(terms, {}) == {"on": "batched", "past": "per_term"}[side]
        elif thr == "terms":
            n = int(side)
            assert len(terms) == n and [len(b) for b in batches] == [32] * (n // 32) + ([n % 32] if n % 32 else [])
        elif thr == "rows":
            g = [t for t in terms if t[0] == "G"]
            assert len(g) == 1 and g[0][1] == int(side) and len(alone) == (int(side) > ops.GLOBAL_ROWS_MAX)
        elif thr == "globalK":
            (t,) = terms
            K = int(side)
            assert t[0] == "G" and t[2] == K
            G_ = max(min(1024 // (K * K), FIN_STAGE_DOUBLES // (K * K)), 1)     # finish.cu global_rows_unit
            assert {22: G_ == 2, 23: G_ == 1, 32: G_ == 1 and K * K == 1024, 33: K * K > 1024, 128: K * K > 1024}[K]
        else:
            raise AssertionError(f"unknown threshold of term set {name}")
    assert seen == {"units32", "e1056", "units16384", "terms", "rows", "globalK"}
    # the automatic per-term route needs no option; the other two routes do not change under the defaults
    assert finish_route(G.TERM_SETS["units16384_past"], {}) == "per_term"
    assert expected_kernels(G.TERM_SETS["units32_on"], {}) == ROUTE_KERNELS["batched"]
