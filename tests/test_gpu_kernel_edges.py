"""Bit-exact probes of every local-IIC kernel family at the edges of its dispatch rule and of its per-CTA work split.

Geometry bugs in these kernels are misrouted, dropped or doubled contributions.  Inputs whose arithmetic is exact in
every kernel's number format expose them with zero tolerance:

* joint probe: one-hot maps (a seeded label per pixel).  Every joint kernel then counts integers exactly (tcj10's
  2^10-scaled fp16 hi part is exact and its lo part 0; tf32 / bf16 hold 0 and 1; per-CTA fp32 partials stay far below
  2^24; the reductions are fp64), so J must EQUAL an int64 count per (dy, dx, i, j), through the reduce launch
  (ops._local_joint) and through iic_finish (ops._finish_terms).
* backward probe: one-hot maps and caller-built coefficients GA[d, i, j] = k * 2^-16 (|k| < 2^16, symmetric in i, j like
  the epilogue's), fed to the raw entry point ops._local_backward_into.  The coefficients have more than 11 significant
  bits, so the fp16 / tf32 lo and correction MMAs carry non-zero values, while every partial sum spans fewer than 24
  bits: each kernel must match the fp64 adjoint bit for bit.  The gradients go into channel-block views of larger
  tensors (NaN inside the block before the call, a sentinel bit pattern outside) whose inputs' neighbouring channels hold
  another one-hot labelling, so a missed store, a store outside the block or a read outside it all break the equality.

Softmax, logs and fp16 rounding of real-valued maps cannot be exact; those cases (from-logits, peaked maps, a map with an
empty cluster) are compared with an fp64 restatement on the device, itself checked against the numpy oracle here, with
the 1e-5 / 1e-4 contract and a tighter bound per family (about 4x the error measured on a B200;
the inputs are seeded, and the from-logits backward varies from call to call only in the last bits):

    case (seeded inputs, deterministic kernels)          largest error measured    bound
    from-logits joint, J (tcj10; fast at W = 244)         1.20e-6 (config-2 size)   5e-6
    from-logits gradients (tcrb10h, seam shapes)          1.72e-6 (H = 3, W = 128)  7e-6
    peaked maps, softmax(8 randn), gradients (tcrb10h)    8.39e-7                   3.5e-6
    one empty cluster, gradients (tcrb10h)                8.88e-7                   3.5e-6

measured on an NVIDIA B200 at its 1000 W power limit.

Which kernel ran is read from torch.profiler (bare function names, as bench.py's count_own_launches parses them); every
case asserts it, and the last test asserts that the module reached exactly the families of FAMILIES.  The shape lists are
functions of the SM count (iic_b200_sm_count) because the dispatch rules and the work split are; test_seam_coverage
(no GPU) shows, for a 148-SM B200, which seam situation each shape is there for.
"""
import contextlib
import os
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_oracle as O  # noqa: E402

# every local kernel family (and the global joint kernels) this module must reach
FAMILIES = {
    "local_joint_tcj10_kernel", "local_joint_fast_kernel", "local_joint_fast7_kernel", "local_joint_tcp_kernel",
    "local_joint_tc_kernel", "local_joint_tma_kernel", "local_joint_kernel",
    "local_bwd_tc_kernel", "local_bwd_tcrb10h_kernel", "local_bwd_tcrb10_kernel", "local_bwd_tcrb_kernel",
    "local_bwd_fast_kernel", "local_bwd_tma_kernel", "local_bwd_kernel",
    "global_joint_kernel", "finish_kernel",
}
JOINT_KERNELS = {f for f in FAMILIES if f.startswith("local_joint")}
BWD_KERNELS = {f for f in FAMILIES if f.startswith("local_bwd")}
_OBSERVED = set()

# per-family error bounds of the tolerance tests (max-norm relative error against fp64), about 4x the B200 measurement
BOUND = {
    "tcj10_logits_joint": 5e-6,
    "tcrb10h_logits": 7e-6,
    "tcrb10h_peaked": 3.5e-6,
    "tcrb10h_zero_channel": 3.5e-6,
}
LOSS_RTOL, GRAD_RTOL = 1e-5, 1e-4
B200_SMS = 148          # the seam list is documented (test_seam_coverage) for this SM count
RMAX = 8                # local_bwd_tcrb10h.cu: output rows per chunk at most
SENTINEL = 0x5A5A5A5A   # a finite float's bit pattern: what must survive outside a gradient block


# ---- seam model (CPU): restatements of the work split; the source of truth is the .cu files ----------------------
def tcrb10h_chunks(B, H, sms):
    """local_bwd_tcrb10h.cu: the B*H rows cut into `sms` CTA shares [R0, R1), each cut by next_chunk into chunks of at
    most RMAX rows.  Returns per chunk (R0, R1, r, n, h0, nr, q0, cont_next)."""
    out = []
    rows = B * H
    for b in range(sms):
        R0, R1 = b * rows // sms, (b + 1) * rows // sms
        share = R1 - R0
        nch = (share + RMAX - 1) // RMAX
        rc = (share + nch - 1) // nch if nch > 0 else RMAX
        r = R0
        while r < R1:
            n, h0 = r // H, r % H
            run = min(H - h0, R1 - r)
            nr = min(rc, run)
            if run - nr == 1 and nr >= 3:
                nr -= 1
            q0 = 2 if (r > R0 and h0 > 0) else 0
            out.append((R0, R1, r, n, h0, nr, q0, nr < run))
            r += nr
    return out


def tcj10_chunks(B, H, sms):
    """local_fwd_tcj10.cu chunk_at: a CTA share [R0, R1) of the B*H rows walked one image at a time; a chunk of nr rows
    is staged as (nr + 1) / 2 row pairs, so an odd nr leaves a single-row pair.  Returns (R0, R1, r, h0, nr)."""
    out = []
    rows = B * H
    for b in range(sms):
        R0, R1 = b * rows // sms, (b + 1) * rows // sms
        r = R0
        while r < R1:
            h0 = r % H
            nr = min(H - h0, R1 - r)
            out.append((R0, R1, r, h0, nr))
            r += nr
    return out


def tcrb10h_cases(s):
    """(B, K, H, W, options, expected kernel) of the K = 9 / 10 tensor-core backward; s = SM count."""
    t = 8 * s
    return [
        (t + 1, 10, 1, 8, {}, "local_bwd_tcrb10h_kernel"),               # H = 1: every chunk one row, shares span images
        (t // 2 + 1, 9, 2, 124, {}, "local_bwd_tcrb10h_kernel"),         # H = 2
        (t // 3 + 1, 10, 3, 128, {}, "local_bwd_tcrb10h_kernel"),        # H = 3: shares start mid-image
        (t // 9 + 1, 9, 9, 132, {}, "local_bwd_tcrb10h_kernel"),         # H = 9: 9-row shares, nr = 1 tail chunks
        (t // 17 + 1, 10, 17, 244, {}, "local_bwd_tcrb10h_kernel"),      # H = 17: shares end inside images
        (9, 10, 224, 224, {}, "local_bwd_tcrb10h_kernel"),               # config-2 size: 7-row chunks, cont_next chains
        (t // 16, 10, 16, 248, {}, "local_bwd_tcrb10h_kernel"),          # widest map, exactly 8 rows per SM
        (t // 16, 10, 16, 252, {}, "local_bwd_fast_kernel"),             # W > 248: falls back
        (t // 16 - 1, 10, 16, 128, {}, "local_bwd_fast_kernel"),         # one image below the row threshold
        (2, 10, 12, 16, {"tc10_force": 1}, "local_bwd_tcrb10h_kernel"),  # forced on a tiny map: 24 rows for every SM, most shares empty
        (9, 10, 224, 224, {"tc10_tf32": 1}, "local_bwd_tcrb10_kernel"),  # tf32 + bf16 form at config-2 size
        (t // 17 + 1, 9, 17, 8, {"tc10_tf32": 1}, "local_bwd_tcrb10_kernel"),
        (t // 3 + 1, 10, 3, 248, {"tc10_tf32": 1}, "local_bwd_tcrb10_kernel"),
    ]


def tcj10_cases(s):
    """(B, K, H, W, expected kernel) of the K <= 10 tensor-core joint; s = SM count."""
    t = 8 * s
    return [
        (t // 8, 10, 8, 8, "local_joint_tcj10_kernel"),          # B*H = 8 SMs exactly
        (t // 8 - 1, 10, 8, 8, "local_joint_fast_kernel"),       # one image below
        (t, 3, 1, 12, "local_joint_tcj10_kernel"),               # H = 1: every share spans 8 images
        (t // 2, 9, 2, 220, "local_joint_tcj10_kernel"),         # H = 2
        (t // 37 + 2, 8, 37, 224, "local_joint_tcj10_kernel"),   # widest map; 8 / 9-row shares ending inside images
        (t // 37 + 2, 2, 37, 228, "local_joint_tma_kernel"),     # W > 224: falls back
        (t // 5 + 3, 2, 5, 16, "local_joint_tcj10_kernel"),      # odd chunks (single-row pairs) inside odd shares
        (t // 13 + 5, 10, 13, 24, "local_joint_tcj10_kernel"),
    ]


# ---- CPU test ----------------------------------------------------------------------------------------------------
def test_seam_coverage():
    """The tensor-core shape lists above reach, on a B200, each situation of the row split they are there for."""
    s = B200_SMS
    seen = set()
    for (B, K, H, W, opts, kern) in tcrb10h_cases(s):
        if kern != "local_bwd_tcrb10h_kernel" or opts:
            continue
        ch = tcrb10h_chunks(B, H, s)
        assert sum(c[5] for c in ch) == B * H and all(1 <= c[5] <= RMAX for c in ch)
        for (R0, R1, r, n, h0, nr, q0, cont) in ch:
            if nr == 1:
                seen.add("nr=1")
            if nr == RMAX:
                seen.add("nr=RMAX")
            if q0 == 2:
                seen.add("q0=2")
            if cont:
                seen.add("cont_next")
            if r == R0 and h0 > 0:
                seen.add("share starts mid-image")
            if (R1 - 1) // H > R0 // H:
                seen.add("share spans images")
            if H < 3:
                seen.add("H<3")
    assert seen == {"nr=1", "nr=RMAX", "q0=2", "cont_next", "share starts mid-image", "share spans images", "H<3"}, seen
    seen = set()
    for (B, K, H, W, kern) in tcj10_cases(s):
        if kern != "local_joint_tcj10_kernel":
            continue
        for (R0, R1, r, h0, nr) in tcj10_chunks(B, H, s):
            if nr % 2:
                seen.add("odd chunk")
            if (R1 - R0) % 2:
                seen.add("odd share")
            if r == R0 and h0 > 0:
                seen.add("share starts mid-image")
            if (R1 - 1) // H > R0 // H:
                seen.add("share spans images")
            if R1 % H:
                seen.add("share ends inside an image")
    assert seen == {"odd chunk", "odd share", "share starts mid-image", "share spans images",
                    "share ends inside an image"}, seen
    # the row threshold at exactly 8 rows per SM and one image below it
    rows = [B * H for (B, K, H, W, kern) in tcj10_cases(s)[:2]]
    assert rows[0] == 8 * s and rows[1] < 8 * s


# ---- GPU helpers ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def iic(cuda_device):
    import iic_b200
    return iic_b200


@pytest.fixture(scope="module")
def sms(iic):
    n = iic._lib.load().iic_b200_sm_count(0)
    assert n > 0
    return n


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
    _OBSERVED.update(names)
    return names


def labels(gen, shape, K, dev):
    return torch.randint(0, K, shape, generator=gen).to(dev)


def onehot(lab, K):
    """(B, H, W) labels, -1 = no cluster -> (B, K, H, W) float32 0 / 1."""
    ok = lab >= 0
    oh = torch.nn.functional.one_hot(lab.clamp(min=0), K).permute(0, 3, 1, 2).float()
    return oh * ok[:, None].float()


def embedded(gen, lab, K, N, C, n0, c0, dev):
    """A channel block [n0:n0+B, c0:c0+K] of an (N, C, H, W) tensor holding onehot(lab); every other channel and
    sample holds another valid one-hot labelling."""
    B, H, W = lab.shape
    full = torch.zeros((N, C, H, W), dtype=torch.float32, device=dev)
    full[:] = onehot(labels(gen, (N, H, W), C, dev), C)
    if C > K:
        rest = [c for c in range(C) if not c0 <= c < c0 + K]
        full[n0:n0 + B, rest] = onehot(labels(gen, (B, H, W), C - K, dev), C - K)
    full[n0:n0 + B, c0:c0 + K] = onehot(lab, K)
    return full, full[n0:n0 + B, c0:c0 + K]


def joint_counts(lx, ly, K, pad):
    """int64 J[dy, dx, i, j] = #{(n, u, v): label_x(n, u+dy-pad, v+dx-pad) = i, label_y(n, u, v) = j}."""
    B, H, W = lx.shape
    T = 2 * pad + 1
    lxp = torch.full((B, H + 2 * pad, W + 2 * pad), -1, dtype=torch.int64, device=lx.device)
    lxp[:, pad:pad + H, pad:pad + W] = lx
    J = torch.empty((T, T, K, K), dtype=torch.int64, device=lx.device)
    for dy in range(T):
        for dx in range(T):
            a = lxp[:, dy:dy + H, dx:dx + W]
            ok = (a >= 0) & (ly >= 0)
            J[dy, dx] = torch.bincount((a * K + ly)[ok], minlength=K * K).view(K, K)
    return J


def adjoint64(x, y, GA, pad):
    """fp64 adjoint of the local joint (oracle local_backward_from_GA on the device); GA (T, T, K, K)."""
    x, y, GA = x.double(), y.double(), GA.double()
    B, K, H, W = x.shape
    T = 2 * pad + 1
    xp = torch.zeros((B, K, H + 2 * pad, W + 2 * pad), dtype=torch.float64, device=x.device)
    xp[:, :, pad:pad + H, pad:pad + W] = x
    gxp, gy = torch.zeros_like(xp), torch.zeros_like(y)
    for dy in range(T):
        for dx in range(T):
            gxp[:, :, dy:dy + H, dx:dx + W] += torch.einsum("ij,njhw->nihw", GA[dy, dx], y)
            gy += torch.einsum("ij,nihw->njhw", GA[dy, dx], xp[:, :, dy:dy + H, dx:dx + W])
    return gxp[:, :, pad:pad + H, pad:pad + W], gy


def joint64(x, y, pad):
    x, y = x.double(), y.double()
    B, K, H, W = x.shape
    T = 2 * pad + 1
    xp = torch.zeros((B, K, H + 2 * pad, W + 2 * pad), dtype=torch.float64, device=x.device)
    xp[:, :, pad:pad + H, pad:pad + W] = x
    return torch.stack([torch.stack([torch.einsum("nihw,njhw->ij", xp[:, :, dy:dy + H, dx:dx + W], y)
                                     for dx in range(T)]) for dy in range(T)])


def exact_coeffs(rng, npatch, K, pad):
    """GA[p, dy, dx, i, j] = k * 2^-16, symmetric in (i, j), |k| < 2^16 (fewer for wide windows, so that a sum over
    T^2 taps stays below 2^24 units of 2^-16)."""
    T = 2 * pad + 1
    kmax = min(2 ** 16, 2 ** 23 // (T * T))
    k = rng.integers(-kmax + 1, kmax, size=(npatch, T, T, K, K))
    k = np.triu(k) + np.swapaxes(np.triu(k, 1), -1, -2)
    return k.astype(np.float64) * 2.0 ** -16


def coeff_buffers(lib, GA, K, pad, dev):
    """Wx / Wy as iic_local_epilogue lays them out (csrc/epilogue.cuh, step 4): [patch][cin][tap][Kp], Kp = K rounded up
    to 4 and zero padded, Wy[i][dy*T+dx][j] = GA[dy, dx, i, j], Wx[j][(T-1-dy)*T+(T-1-dx)][i] = GA[dy, dx, i, j]; then
    the scratch tail of iic_local_coeff_floats floats the tensor-core kernels build their weight image in."""
    npatch, T = GA.shape[0], 2 * pad + 1
    Kp = (K + 3) & ~3
    wy = np.zeros((npatch, K, T * T, Kp))
    wx = np.zeros((npatch, K, T * T, Kp))
    for dy in range(T):
        for dx in range(T):
            wy[:, :, dy * T + dx, :K] = GA[:, dy, dx]
            wx[:, :, (T - 1 - dy) * T + (T - 1 - dx), :K] = np.swapaxes(GA[:, dy, dx], -1, -2)
    n = lib.iic_local_coeff_floats(K, pad, npatch)
    out = []
    for w in (wx, wy):
        b = torch.zeros(n, dtype=torch.float32)
        b[:w.size] = torch.from_numpy(w.reshape(-1).astype(np.float32))
        out.append(b.to(dev))
    return out


def grad_block(N, C, n0, c0, B, K, H, W, dev, fill):
    G = torch.empty((N, C, H, W), dtype=torch.float32, device=dev)
    G.view(torch.int32).fill_(SENTINEL)
    G[n0:n0 + B, c0:c0 + K] = fill
    return G, G[n0:n0 + B, c0:c0 + K]


def assert_outside_untouched(G, n0, c0, B, K):
    bits = G.view(torch.int32).clone()
    bits[n0:n0 + B, c0:c0 + K] = SENTINEL
    bad = (bits != SENTINEL).nonzero()
    assert bad.numel() == 0, f"{bad.shape[0]} elements written outside the block, first at {bad[0].tolist()}"


def first_mismatch(a, b):
    d = (a.double() != b.double()).nonzero()
    if d.numel() == 0:
        return "none"
    i = tuple(d[0].tolist())
    return f"{d.shape[0]} entries differ, first at {i}: {a[i].item()!r} vs {b[i].item()!r}"


# ---- exact joint probe -----------------------------------------------------------------------------------------
def _joint_case(iic, dev, B, K, H, W, pad, expect, opts=None, mask=False, patch=None, block=None, seed=0):
    gen = torch.Generator().manual_seed(seed)
    lx, ly = labels(gen, (B, H, W), K, dev), labels(gen, (B, H, W), K, dev)
    m = None
    if mask:
        # the maps keep their labels under the mask's zeros: the kernel has to apply the mask itself
        mk = torch.rand((B, 1, H, W), generator=gen).to(dev) < 0.7
        m = mk.float()
        x, y = onehot(lx, K), onehot(ly, K)
        lx, ly = torch.where(mk[:, 0], lx, -1), torch.where(mk[:, 0], ly, -1)
    elif block:
        N, C, n0, c0 = block
        _, x = embedded(gen, lx, K, N, C, n0, c0, dev)
        _, y = embedded(gen, ly, K, N, C, n0, c0, dev)
    else:
        x, y = onehot(lx, K), onehot(ly, K)
    ph, pw, sh, sw = patch if patch else (H, W, H, W)
    wins = O.patch_windows(H, W, (ph, pw), (sh, sw))
    ref = torch.stack([joint_counts(lx[:, h0:h1, w0:w1], ly[:, h0:h1, w0:w1], K, pad) for (h0, h1, w0, w1) in wins])
    with options(iic, opts or {}):
        out = {}
        ks = kernels(lambda: out.setdefault("J", iic.ops._local_joint(x, y, m, pad, ph, pw, sh, sw)))
        term = iic.ops.LocalTerm(x, y, m, pad, (ph, pw), (sh, sw), 1.0)
        kf = kernels(lambda: out.setdefault("F", iic.ops._finish_terms([term], False)[0]["J"]))
    assert expect in ks and not (ks & JOINT_KERNELS) - {expect}, ks
    assert expect in kf and "finish_kernel" in kf, kf
    J, JF = out["J"], out["F"].view(ref.shape)
    assert torch.equal(J, ref.double()), first_mismatch(J, ref)
    assert torch.equal(JF, ref.double()), first_mismatch(JF, ref)


def _joint_matrix(s):
    t = 8 * s
    cases = [(B, K, H, W, 1, kern, {}, {}) for (B, K, H, W, kern) in tcj10_cases(s)]
    cases += [
        (t // 8, 10, 8, 24, 1, "local_joint_tcj10_kernel", {}, {"block": (t // 8 + 3, 16, 2, 6)}),   # c0 + K == C
        (t // 8, 7, 8, 16, 1, "local_joint_tcj10_kernel", {}, {"block": (t // 8 + 1, 12, 1, 2)}),
        (t // 8, 10, 8, 8, 1, "local_joint_fast_kernel", {"no_tcj10": 1}, {}),
        (2, 10, 12, 16, 1, "local_joint_fast_kernel", {}, {}),
        (2, 16, 20, 300, 1, "local_joint_fast_kernel", {}, {}),                    # K % 8 blocks, wide map
        (2, 20, 40, 64, 3, "local_joint_tcp_kernel", {}, {}),                      # packed tensor-core joint, padding 3
        (3, 24, 9, 48, 3, "local_joint_tcp_kernel", {}, {"block": (4, 30, 1, 6)}),
        (2, 16, 12, 64, 1, "local_joint_tcp_kernel", {"tcp_p1": 1}, {}),
        (2, 20, 16, 36, 3, "local_joint_fast7_kernel", {}, {}),                    # W % 16 != 0: two 10-channel slabs
        (1, 10, 40, 260, 3, "local_joint_fast7_kernel", {}, {}),
        (1, 128, 24, 32, 1, "local_joint_tc_kernel", {}, {}),
        (1, 128, 8, 20, 1, "local_joint_fast_kernel", {}, {}),                     # W % 16 != 0: blocks of 8
        (2, 3, 12, 16, 1, "local_joint_tma_kernel", {}, {}),
        (2, 5, 9, 20, 2, "local_joint_tma_kernel", {}, {}),
        (2, 6, 11, 13, 1, "local_joint_kernel", {}, {}),                           # W % 4 != 0
        (2, 6, 14, 18, 1, "local_joint_kernel", {}, {"mask": True}),
        (2, 5, 20, 24, 1, "local_joint_kernel", {}, {"patch": (8, 8, 4, 4)}),     # overlapping patches
        (2, 4, 9, 11, 0, "local_joint_kernel", {"no_tma": 1}, {}),
        (1, 3, 12, 10, 4, "local_joint_kernel", {}, {}),
        (1, 2, 5, 7, 7, "local_joint_kernel", {}, {}),
    ]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(_joint_matrix(B200_SMS))))
def test_joint_exact(iic, cuda_device, sms, idx):
    B, K, H, W, pad, kern, opts, kw = _joint_matrix(sms)[idx]
    _joint_case(iic, cuda_device, B, K, H, W, pad, kern, opts, seed=idx, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("N,K", [(64, 10), (4096, 20), (4097, 10), (70000, 16)])
def test_global_joint_exact(iic, cuda_device, N, K):
    dev = cuda_device
    gen = torch.Generator().manual_seed(N)
    lx, ly = labels(gen, (N,), K, dev), labels(gen, (N,), K, dev)
    x = torch.nn.functional.one_hot(lx, K).float()
    y = torch.nn.functional.one_hot(ly, K).float()
    ref = torch.bincount(lx * K + ly, minlength=K * K).view(K, K).double()
    out = {}
    if N <= iic.ops.GLOBAL_ROWS_MAX:
        ks = kernels(lambda: out.setdefault("J", iic.ops._finish_terms([iic.ops.GlobalTerm(x, y)], False)[0]["J"]))
        assert "finish_kernel" in ks, ks
    else:
        ks = kernels(lambda: out.setdefault("J", iic.ops._global_joint(x, y)))
        assert "global_joint_kernel" in ks, ks
    J = out["J"].view(K, K)
    assert torch.equal(J, ref), first_mismatch(J, ref)


# ---- exact backward probe, write coverage and confinement ------------------------------------------------------
def _bwd_case(iic, dev, B, K, H, W, pad, expect, opts=None, mask=False, patch=None, block=None, g=1.0, seed=0):
    lib = iic._lib.load()
    gen = torch.Generator().manual_seed(1000 + seed)
    rng = np.random.default_rng(seed)
    lx, ly = labels(gen, (B, H, W), K, dev), labels(gen, (B, H, W), K, dev)
    N, C, n0, c0 = block if block else (B + 2, K + 3, 1, 3)
    _, x = embedded(gen, lx, K, N, C, n0, c0, dev)
    _, y = embedded(gen, ly, K, N, C, n0, c0, dev)
    m = None
    if mask:
        m = (torch.rand((B, 1, H, W), generator=gen) < 0.7).float().to(dev)
    ph, pw, sh, sw = patch if patch else (H, W, H, W)
    wins = O.patch_windows(H, W, (ph, pw), (sh, sw))
    GA = exact_coeffs(rng, len(wins), K, pad)
    Wx, Wy = coeff_buffers(lib, GA, K, pad, dev)
    GAd = torch.from_numpy(GA).to(dev)
    xm, ym = (x, y) if m is None else (x * m, y * m)
    rx = torch.zeros((B, K, H, W), dtype=torch.float64, device=dev)
    ry = torch.zeros_like(rx)
    for p, (h0, h1, w0, w1) in enumerate(wins):
        a, b = adjoint64(xm[:, :, h0:h1, w0:w1], ym[:, :, h0:h1, w0:w1], GAd[p], pad)
        rx[:, :, h0:h1, w0:w1] += a
        ry[:, :, h0:h1, w0:w1] += b
    if m is not None:
        rx, ry = rx * m, ry * m
    rx, ry = rx * g, ry * g
    fill = 0.0 if len(wins) > 1 else float("nan")          # several patches accumulate into zero-filled gradients
    Gx, gx = grad_block(N, C, n0, c0, B, K, H, W, dev, fill)
    Gy, gy = grad_block(N, C, n0, c0, B, K, H, W, dev, fill)
    grad = torch.tensor(g, dtype=torch.float32, device=dev)
    with options(iic, opts or {}):
        ks = kernels(lambda: iic.ops._local_backward_into(x, y, m, Wx, Wy, grad, pad, ph, pw, sh, sw, gx, gy))
    assert expect in ks and not (ks & BWD_KERNELS) - {expect}, ks
    for name, G, gv, r in (("gx", Gx, gx, rx), ("gy", Gy, gy, ry)):
        nan = torch.isnan(gv)
        assert not nan.any(), f"{name}: {int(nan.sum())} elements never written, first at {nan.nonzero()[0].tolist()}"
        assert torch.equal(gv.double(), r), f"{name}: {first_mismatch(gv, r)}"
        assert_outside_untouched(G, n0, c0, B, K)


def _bwd_matrix(s):
    cases = [(B, K, H, W, 1, kern, opts, {}) for (B, K, H, W, opts, kern) in tcrb10h_cases(s)]
    cases += [
        (9, 10, 224, 224, 1, "local_bwd_tcrb10h_kernel", {}, {"g": -0.5, "block": (10, 10, 1, 0)}),   # c0 = 0
        (3 * s, 9, 3, 64, 1, "local_bwd_tcrb10h_kernel", {}, {"block": (3 * s + 1, 13, 0, 4)}),       # c0 + K == C
        (2, 20, 40, 64, 3, "local_bwd_tcrb_kernel", {}, {}),                     # padding 3
        (1, 24, 20, 300, 3, "local_bwd_tcrb_kernel", {}, {"g": -0.5}),           # two 152-column panels, the last one ragged
        (1, 16, 12, 512, 3, "local_bwd_tcrb_kernel", {}, {}),                    # four 128-column panels
        (2 * s, 16, 1, 128, 1, "local_bwd_tcrb_kernel", {}, {}),                 # padding 1: n_items == 2 SMs
        (2 * s - 1, 16, 1, 128, 1, "local_bwd_fast_kernel", {}, {}),             # one item below
        (2, 20, 10, 64, 1, "local_bwd_tcrb_kernel", {"tcrb_p1": 1}, {"block": (3, 20, 1, 0)}),
        (1, 128, 8, 8, 1, "local_bwd_tc_kernel", {}, {}),
        (1, 128, 7, 16, 1, "local_bwd_tc_kernel", {}, {"block": (2, 130, 1, 2)}),
        (1, 128, 6, 248, 1, "local_bwd_tc_kernel", {}, {"g": -0.5}),
        (2, 10, 12, 16, 1, "local_bwd_fast_kernel", {}, {}),
        (1, 10, 6, 300, 1, "local_bwd_fast_kernel", {}, {}),                     # two 152-column panels
        (2, 20, 16, 36, 3, "local_bwd_fast_kernel", {"no_tc": 1}, {}),           # padding 3, two 10-channel blocks
        (1, 8, 10, 500, 3, "local_bwd_fast_kernel", {"no_tc": 1}, {"g": -0.5}),
        (2, 3, 12, 16, 1, "local_bwd_tma_kernel", {}, {}),
        (2, 5, 9, 20, 0, "local_bwd_tma_kernel", {}, {}),
        (2, 6, 11, 13, 1, "local_bwd_kernel", {}, {}),                           # W % 4 != 0, odd strides
        (2, 6, 14, 16, 1, "local_bwd_kernel", {}, {"mask": True}),
        (2, 5, 20, 24, 1, "local_bwd_kernel", {}, {"patch": (8, 8, 4, 4)}),     # overlapping patches accumulate
        (2, 4, 9, 12, 0, "local_bwd_kernel", {"no_tma": 1}, {}),
        (1, 3, 12, 10, 2, "local_bwd_kernel", {}, {"g": -0.5}),
        (1, 3, 12, 10, 4, "local_bwd_kernel", {}, {}),
        (1, 2, 5, 7, 7, "local_bwd_kernel", {}, {}),
    ]
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("idx", range(len(_bwd_matrix(B200_SMS))))
def test_backward_exact(iic, cuda_device, sms, idx):
    B, K, H, W, pad, kern, opts, kw = _bwd_matrix(sms)[idx]
    _bwd_case(iic, cuda_device, B, K, H, W, pad, kern, opts, seed=idx, **kw)


@pytest.mark.gpu
def test_coefficient_layout_matches_epilogue(iic, cuda_device):
    """coeff_buffers restates the layout iic_local_epilogue writes: both agree on a real joint to fp32 rounding."""
    dev = cuda_device
    lib = iic._lib.load()
    rng = np.random.default_rng(5)
    for (K, pad) in ((10, 1), (5, 2)):
        x = torch.from_numpy(O.softmax(rng.standard_normal((2, K, 12, 16)) * 2).astype(np.float32)).to(dev)
        y = torch.from_numpy(O.softmax(rng.standard_normal((2, K, 12, 16)) * 2).astype(np.float32)).to(dev)
        J = iic.ops._local_joint(x, y, None, pad, 12, 16, 12, 16)
        _, Wx, Wy = iic.ops._local_epilogue(J, K, pad, 1.0)
        GA = O.local_loss_from_joint(J[0].cpu().numpy())[1]
        hx, hy = coeff_buffers(lib, GA[None], K, pad, dev)
        n = (2 * pad + 1) ** 2 * K * ((K + 3) & ~3)
        for a, b in ((Wx, hx), (Wy, hy)):
            a, b = a[:n].double(), b[:n].double()
            assert ((a - b).abs() <= 2e-7 * b.abs().max()).all(), (a - b).abs().max().item()


@pytest.mark.gpu
def test_torch_restatement_matches_oracle(cuda_device):
    """joint64 / adjoint64 (the fp64 references of the tolerance tests) against the numpy oracle."""
    rng = np.random.default_rng(3)
    x, y = O.softmax(rng.standard_normal((2, 4, 9, 11))), O.softmax(rng.standard_normal((2, 4, 9, 11)))
    J = O.local_joint(x, y, 2)
    GA = O.local_loss_from_joint(J)[1]
    ogx, ogy = O.local_backward_from_GA(x, y, GA, 2)
    xd, yd = torch.from_numpy(x).to(cuda_device), torch.from_numpy(y).to(cuda_device)
    assert np.allclose(joint64(xd, yd, 2).cpu().numpy(), J, rtol=1e-13, atol=0)
    gx, gy = adjoint64(xd, yd, torch.from_numpy(GA).to(cuda_device), 2)
    assert np.allclose(gx.cpu().numpy(), ogx, rtol=1e-12, atol=1e-15)
    assert np.allclose(gy.cpu().numpy(), ogy, rtol=1e-12, atol=1e-15)


# ---- confinement of the from-logits and global backwards --------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape_idx", [0, 4, 5])
def test_from_logits_backward_confined(iic, cuda_device, sms, shape_idx):
    """The from-logits backward writes its channel block of a larger gradient tensor completely and nothing else.  Its
    result is compared with fp64, not bit for bit: where row chunks chain (H > 1) two identical calls already differ
    in the last bits."""
    dev = cuda_device
    B, K, H, W, _, kern = tcrb10h_cases(sms)[shape_idx]
    gen = torch.Generator().manual_seed(11)
    N, C, n0, c0 = B + 1, K + 5, 1, 2
    L = torch.randn((N, C, H, W), generator=gen).to(dev) * 2
    lx, ly = L[n0:n0 + B, c0:c0 + K], (L * 0.8 + 0.1)[n0:n0 + B, c0:c0 + K]
    J = iic.ops._local_joint_logits(lx, ly, 1, 1.0)
    _, Wx, Wy = iic.ops._local_epilogue(J, K, 1, 1.0)
    grad = torch.tensor(1.0, device=dev)
    Gx, gx = grad_block(N, C, n0, c0, B, K, H, W, dev, float("nan"))
    Gy, gy = grad_block(N, C, n0, c0, B, K, H, W, dev, float("nan"))
    ks = kernels(lambda: iic.ops._local_backward_logits_into(lx, ly, Wx, Wy, grad, 1, 1.0, gx, gy))
    assert kern in ks, ks
    _, _, rx, ry = _logits_reference(lx, ly)
    for name, G, gv, ref in (("gx", Gx, gx, rx), ("gy", Gy, gy, ry)):
        nan = torch.isnan(gv)
        assert not nan.any(), f"{name}: {int(nan.sum())} elements never written, first at {nan.nonzero()[0].tolist()}"
        _grad_err(gv, ref, sms, f"from-logits block ({B},{K},{H},{W}) {name}", BOUND["tcrb10h_logits"])
        assert_outside_untouched(G, n0, c0, B, K)


@pytest.mark.gpu
@pytest.mark.parametrize("N,K,C,c0", [(1000, 10, 16, 6), (5000, 20, 23, 1), (333, 7, 9, 0)])
def test_global_backward_confined(iic, cuda_device, N, K, C, c0):
    dev = cuda_device
    gen = torch.Generator().manual_seed(N)
    x = torch.softmax(torch.randn((N, K), generator=gen) * 2, 1).to(dev)
    y = torch.softmax(torch.randn((N, K), generator=gen) * 2, 1).to(dev)
    J = iic.ops._global_joint(x, y)
    gl, gn = torch.tensor(1.0, device=dev), torch.tensor(-0.5, device=dev)
    dx, dy = iic.ops._global_backward(x, y, J, 1.0, True, gl, gn, None)
    out = []
    for _ in range(2):
        G = torch.empty((N, C), dtype=torch.float32, device=dev)
        G.view(torch.int32).fill_(SENTINEL)
        G[:, c0:c0 + K] = float("nan")
        out.append(G)
    iic.ops._global_backward_into(x, y, J, 1.0, True, gl, gn, None, out[0][:, c0:c0 + K], out[1][:, c0:c0 + K])
    for G, ref in zip(out, (dx, dy)):
        assert torch.equal(G[:, c0:c0 + K], ref), first_mismatch(G[:, c0:c0 + K], ref)
        bits = G.view(torch.int32).clone()
        bits[:, c0:c0 + K] = SENTINEL
        assert (bits == SENTINEL).all()


# ---- tolerance tests where exactness is impossible -------------------------------------------------------------
def regions(err, sms):
    """Largest relative error per region of a (B, K, H, W) error map: first / last image row, rows at CTA share
    boundaries, first / last column, the last 32-column tile, and each channel."""
    B, K, H, W = err.shape
    rows = err.permute(0, 2, 1, 3).reshape(B * H, K, W)
    bnd = sorted({b * B * H // sms for b in range(1, sms)} | {b * B * H // sms - 1 for b in range(1, sms)})
    out = {"first row": err[:, :, 0].max(), "last row": err[:, :, -1].max(), "share edges": rows[bnd].max(),
           "first col": err[..., 0].max(), "last col": err[..., -1].max(), "last tile": err[..., -32:].max()}
    out.update({f"ch{k}": err[:, k].max() for k in range(K)})
    return {k: float(v) for k, v in out.items()}


def _grad_err(g, ref, sms, what, bound):
    scale = ref.abs().max()
    err = (g.double() - ref).abs() / scale
    e = float(err.max())
    print(f"{what}: grad relmax {e:.3e} (bound {bound:.1e})")
    assert e <= min(bound, GRAD_RTOL), (what, e, regions(err, sms))
    return e


def _prob_case(iic, dev, sms, x, y, what, bound):
    B, K, H, W = x.shape
    J = iic.ops._local_joint(x, y, None, 1, H, W, H, W)
    loss, Wx, Wy = iic.ops._local_epilogue(J, K, 1, 1.0)
    grad = torch.tensor(1.0, device=dev)
    gx = torch.empty_like(x)
    gy = torch.empty_like(y)
    ks = kernels(lambda: iic.ops._local_backward_into(x, y, None, Wx, Wy, grad, 1, H, W, H, W, gx, gy))
    assert "local_bwd_tcrb10h_kernel" in ks, ks
    J64 = joint64(x, y, 1)
    ol, GA = O.local_loss_from_joint(J64.cpu().numpy())
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol), (loss.item(), ol)
    rx, ry = adjoint64(x, y, torch.from_numpy(GA).to(dev), 1)
    return max(_grad_err(gx, rx, sms, what + " gx", bound), _grad_err(gy, ry, sms, what + " gy", bound))


def _logits_reference(lx, ly):
    """fp64 joint, loss and logit gradients of the from-logits local term (padding 1, lamda 1, temperature 1)."""
    px, py = torch.softmax(lx.double(), 1), torch.softmax(ly.double(), 1)
    J64 = joint64(px, py, 1)
    ol, GA = O.local_loss_from_joint(J64.cpu().numpy())
    ax, ay = adjoint64(px, py, torch.from_numpy(GA).to(lx.device), 1)
    rx = px * (ax - (ax * px).sum(1, keepdim=True))            # softmax adjoint
    ry = py * (ay - (ay * py).sum(1, keepdim=True))
    return J64, ol, rx, ry


@pytest.mark.gpu
@pytest.mark.parametrize("shape_idx", [0, 2, 4, 5])
def test_from_logits_tensor_core_tolerance(iic, cuda_device, sms, shape_idx):
    """From-logits tcj10 joint and tcrb10h backward at the seam shapes against fp64."""
    dev = cuda_device
    B, K, H, W, _, _ = tcrb10h_cases(sms)[shape_idx]
    gen = torch.Generator().manual_seed(21 + shape_idx)
    lx = (torch.randn((B, K, H, W), generator=gen) * 2).to(dev)
    ly = (lx + torch.randn((B, K, H, W), generator=gen).to(dev)).contiguous()
    out = {}
    ks = kernels(lambda: out.setdefault("J", iic.ops._local_joint_logits(lx, ly, 1, 1.0)))
    if W <= 224:
        assert "local_joint_tcj10_kernel" in ks, ks
    J64, ol, rx, ry = _logits_reference(lx, ly)
    ej = float((out["J"][0] - J64).abs().max() / J64.abs().max())
    print(f"from-logits joint ({B},{K},{H},{W}): J relmax {ej:.3e}")
    assert ej <= BOUND["tcj10_logits_joint"], ej
    loss, Wx, Wy = iic.ops._local_epilogue(out["J"], K, 1, 1.0)
    grad = torch.tensor(1.0, device=dev)
    gx, gy = torch.empty_like(lx), torch.empty_like(ly)
    kb = kernels(lambda: iic.ops._local_backward_logits_into(lx, ly, Wx, Wy, grad, 1, 1.0, gx, gy))
    assert "local_bwd_tcrb10h_kernel" in kb, kb
    assert abs(loss.item() - ol) <= LOSS_RTOL * abs(ol), (loss.item(), ol)
    _grad_err(gx, rx, sms, f"from-logits ({B},{K},{H},{W}) gx", BOUND["tcrb10h_logits"])
    _grad_err(gy, ry, sms, f"from-logits ({B},{K},{H},{W}) gy", BOUND["tcrb10h_logits"])


@pytest.mark.gpu
def test_peaked_maps_tensor_core_tolerance(iic, cuda_device, sms):
    dev = cuda_device
    B, K, H, W = 9, 10, 224, 224
    gen = torch.Generator().manual_seed(31)
    base = torch.randn((B, K, H // 8, W // 8), generator=gen).repeat_interleave(8, 2).repeat_interleave(8, 3)
    x = torch.softmax(8 * (base + 0.3 * torch.randn((B, K, H, W), generator=gen)), 1).to(dev)
    y = torch.softmax(8 * (base + 0.3 * torch.randn((B, K, H, W), generator=gen)), 1).to(dev)
    _prob_case(iic, dev, sms, x, y, "peaked", BOUND["tcrb10h_peaked"])


@pytest.mark.gpu
def test_empty_cluster_tensor_core_tolerance(iic, cuda_device, sms):
    """One cluster channel identically zero: its joint row and column vanish, so the epilogue's coefficients are the
    largest it produces (log of eps), which exercises the fp16 coefficient scaling of tcrb10h."""
    dev = cuda_device
    B, K, H, W = 9, 10, 224, 224
    gen = torch.Generator().manual_seed(41)
    base = torch.randn((B, K, H // 8, W // 8), generator=gen).repeat_interleave(8, 2).repeat_interleave(8, 3)
    maps = []
    for _ in range(2):
        p = torch.softmax(3 * (base + 0.5 * torch.randn((B, K, H, W), generator=gen)), 1)
        p[:, 3] = 0
        maps.append((p / p.sum(1, keepdim=True)).to(dev))
    _prob_case(iic, dev, sms, maps[0], maps[1], "empty cluster", BOUND["tcrb10h_zero_channel"])


# ---- every switch changes the kernel ----------------------------------------------------------------------------
def _switch_cases(s):
    t = 8 * s
    return {
        # switch: (kind, B, K, H, W, pad)
        "no_tma": ("joint", 2, 10, 12, 16, 1),
        "no_tc": ("joint", 2, 20, 40, 64, 3),
        "no_tc10": ("bwd", t + 1, 10, 1, 8, 1),
        "no_fast": ("joint", 2, 10, 12, 16, 1),
        "tcp_p1": ("joint", 2, 16, 12, 64, 1),
        "tcrb_p1": ("bwd", 2, 16, 8, 64, 1),
        "tc10_force": ("bwd", 2, 10, 12, 16, 1),
        "no_tcj10": ("joint", t // 8, 10, 8, 8, 1),
        "tc10_tf32": ("bwd", t + 1, 10, 1, 8, 1),
        "no_fused_epilogue": ("finish", 2, 10, 12, 16, 1),
        "fin_last_cta_epilogue": ("finish", 2, 10, 12, 16, 1),
    }


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(_switch_cases(B200_SMS)))
def test_switch_changes_kernel(iic, cuda_device, sms, name):
    """Every dispatch switch of iic_b200_set_option selects other kernels on a shape it applies to.  (xchg_timeout_ms is
    a timeout, not a kernel switch.)"""
    dev = cuda_device
    kind, B, K, H, W, pad = _switch_cases(sms)[name]
    gen = torch.Generator().manual_seed(7)
    x = torch.softmax(torch.randn((B, K, H, W), generator=gen), 1).to(dev)
    y = torch.softmax(torch.randn((B, K, H, W), generator=gen), 1).to(dev)
    if kind == "bwd":
        _, Wx, Wy = iic.ops._local_epilogue(iic.ops._local_joint(x, y, None, pad, H, W, H, W), K, pad, 1.0)
        grad = torch.tensor(1.0, device=dev)
        gx, gy = torch.empty_like(x), torch.empty_like(y)
        fn = lambda: iic.ops._local_backward_into(x, y, None, Wx, Wy, grad, pad, H, W, H, W, gx, gy)  # noqa: E731
    elif kind == "joint":
        fn = lambda: iic.ops._local_joint(x, y, None, pad, H, W, H, W)  # noqa: E731
    else:
        fn = lambda: iic.ops._finish_terms([iic.ops.LocalTerm(x, y, None, pad, (H, W), (H, W), 1.0)], False)  # noqa: E731
    with options(iic, {name: 0}):
        off = kernels(fn)
    with options(iic, {name: 1}):
        on = kernels(fn)
    print(f"{name}: off {sorted(off)} on {sorted(on)}")
    assert off != on, (name, off)


@pytest.mark.gpu
def test_every_family_reached(request):
    """Closing check: over this module the profiler saw exactly the families of FAMILIES (the module's tests must run
    before this one, in file order)."""
    ran = {i.name for i in request.session.items if i.module is request.module}
    need = {f"test_joint_exact[{i}]" for i in range(len(_joint_matrix(B200_SMS)))}
    need |= {f"test_backward_exact[{i}]" for i in range(len(_bwd_matrix(B200_SMS)))}
    if not need <= ran:
        pytest.skip("only part of the module was selected")
    assert _OBSERVED & (JOINT_KERNELS | BWD_KERNELS | {"global_joint_kernel", "finish_kernel"}) == FAMILIES, \
        sorted(FAMILIES ^ (_OBSERVED & (JOINT_KERNELS | BWD_KERNELS | {"global_joint_kernel", "finish_kernel"})))
