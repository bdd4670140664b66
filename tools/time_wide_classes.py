"""Times the wide-class (9 <= C <= 256) UDA, supervised and flip-aligned losses, forward + backward, against the
reference's formulas in eager torch on the same GPU, and the supervised loss with an ignore label for 4 to 150 classes.

    python tools/time_wide_classes.py [--reps N] [--losses sup,sup_ignore,...]

Fused: one CUDA graph per workload (forward and backward of the library's loss).  Eager: the reference's composition,
  UDA        softmax of both maps, then the KL_div expression (semi_seg/epocher.py:221-224; kl_losses.py:107-126)
             or torch.nn.MSELoss;
  supervised F.one_hot(long), the KL_div expression, logits.max(1)[1] and the one-hot Dice sums
             (epocher.py:165-166,183-184);
  sup_ignore the supervised loss with ignore_index=255 on Cityscapes-style labels (10 % of the pixels void); eager:
             F.cross_entropy(ignore_index=255), logits.max(1)[1] and the Dice sums of the one-hots masked to the kept
             pixels;
  flip       the per-sample flip loop and torch.stack (epocher.py:160-161), then the UDA term.
Each pass streams from HBM: the input maps of the wide shapes are larger than the 126 MB L2, and a shape whose working
set is smaller is timed round-robin over enough copies of its inputs that a pass never finds its data in L2.
Algorithmic bytes per pixel: 20*C for UDA (forward reads 2C floats, backward reads 2C and writes C), 12*C + 16 for
supervised with or without the ignore label (forward reads C floats and an int64 label, backward reads the same and
writes C).  The HBM peak is measured in the same run with a device-to-device copy; the card's name and power limit are
printed beside it.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import iic_b200  # noqa: E402

SHAPES = [("cityscapes", (16, 19, 512, 1024)), ("voc", (16, 21, 512, 512)), ("ade", (8, 150, 256, 256)),
          ("narrow", (32, 4, 224, 224))]
NARROW_LOSSES = ("sup", "sup_ignore")         # the C <= 8 kernels of the other losses are timed by bench.py
EPS = 1e-16
IGNORE = 255
L2_BYTES = 126 << 20


def timed(fns, reps, min_window_ms=200.0):
    """Mean time of one call, cycling through `fns` (one per copy of the inputs), over at least `reps` calls and a
    window of at least `min_window_ms`."""
    for f in fns:
        f()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while True:
        a.record()
        for i in range(reps):
            fns[i % len(fns)]()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        if ms >= min_window_ms:
            return ms / reps
        reps = int(reps * min_window_ms / max(ms, 1e-3)) + 1


def graphed(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        fn()
    return g.replay


def power_limit():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip() or "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown"


def hbm_peak(dev, reps):
    n = 1 << 30                                                 # 4 GiB per buffer
    src = torch.empty(n, dtype=torch.float32, device=dev).fill_(1.0)
    dst = torch.empty_like(src)
    ms = timed([lambda: dst.copy_(src)], reps)
    del src, dst
    return 2 * 4 * n / (ms * 1e-3)


def uda_eager(s, t, kind):
    p, q = s.softmax(1), t.softmax(1).detach()
    if kind == "kl":
        loss = (-q * torch.log((p + EPS) / (q + EPS))).sum(1).mean()
    else:
        loss = F.mse_loss(p, q)
    return torch.autograd.grad(loss, s)


def sup_eager(lg, lab, C):
    p = lg.softmax(1)
    oh = F.one_hot(lab, C).permute(0, 3, 1, 2)
    loss = (-oh * torch.log((p + EPS) / (oh + EPS))).sum(1).mean()
    pred = F.one_hot(lg.detach().max(1)[1], C).permute(0, 3, 1, 2)
    inter, union = (pred * oh).sum((2, 3)), (pred + oh).sum((2, 3))
    return torch.autograd.grad(loss, lg), inter, union


def sup_ignore_eager(lg, lab, C):
    loss = F.cross_entropy(lg, lab, ignore_index=IGNORE)
    keep = (lab != IGNORE).unsqueeze(1)
    oh = F.one_hot(lab.masked_fill(lab == IGNORE, 0), C).permute(0, 3, 1, 2) * keep
    pred = F.one_hot(lg.detach().max(1)[1], C).permute(0, 3, 1, 2) * keep
    inter, union = (pred * oh).sum((2, 3)), (pred + oh).sum((2, 3))
    return torch.autograd.grad(loss, lg), inter, union


def flip_eager(s, t, flags, kind):
    def T(x, f):
        x = x.clone()
        if f & 1:
            x = x.flip(1)
        if f & 2:
            x = x.flip(2)
        return x
    tf = torch.stack([T(x, int(f)) for x, f in zip(t, flags)], dim=0)
    return uda_eager(s, tf, kind)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--losses", default="uda_kl,uda_mse,sup,sup_ignore,flip_kl")
    args = ap.parse_args()
    losses = args.losses.split(",")
    if not torch.cuda.is_available():
        raise SystemExit("time_wide_classes.py needs a CUDA device")
    dev = torch.device("cuda:0")
    iic_b200.set_check_mode("deferred")
    card = torch.cuda.get_device_name(dev)
    peak = hbm_peak(dev, args.reps)
    print(f"card: {card}, power limit: {power_limit()}, measured HBM copy peak: {peak / 1e12:.2f} TB/s")
    rows = []
    for name, (B, C, H, W) in SHAPES:
        names = [w for w in losses if C > 8 or w in NARROW_LOSSES]
        if not names:
            continue
        npx = B * H * W
        # copies of the inputs so that one round-robin cycle moves more than twice the L2 (the largest workload's
        # working set is 12*C + 16 bytes per pixel for supervised, 20*C for UDA)
        ncopy = max(1, -(-2 * L2_BYTES // (12 * C + 16) // npx))
        g = torch.Generator(device=dev).manual_seed(C)
        sets = []
        for _ in range(ncopy):
            s = (torch.randn(B, C, H, W, device=dev, generator=g) * 2).requires_grad_(True)
            t = torch.randn(B, C, H, W, device=dev, generator=g) * 2 if C > 8 else None
            lab = torch.randint(0, C, (B, H, W), device=dev, generator=g)
            void = lab.masked_fill(torch.rand(B, H, W, device=dev, generator=g) < 0.1, IGNORE)
            sets.append((s, t, lab, void))
        flags = torch.arange(B, dtype=torch.uint8) % 4
        flags_dev = flags.to(dev)

        def work(wname, s, t, lab, void):
            return {
                "uda_kl": (lambda: torch.autograd.grad(iic_b200.uda_from_logits(s, t, "kl"), s),
                           lambda: uda_eager(s, t, "kl"), 20 * C),
                "uda_mse": (lambda: torch.autograd.grad(iic_b200.uda_from_logits(s, t, "mse"), s),
                            lambda: uda_eager(s, t, "mse"), 20 * C),
                "sup": (lambda: torch.autograd.grad(iic_b200.sup_kl_from_logits(s, lab, return_dice=True)[0], s),
                        lambda: sup_eager(s, lab, C), 12 * C + 16),
                "sup_ignore": (lambda: torch.autograd.grad(
                                   iic_b200.sup_kl_from_logits(s, void, return_dice=True, ignore_index=IGNORE)[0], s),
                               lambda: sup_ignore_eager(s, void, C), 12 * C + 16),
                "flip_kl": (lambda: torch.autograd.grad(iic_b200.uda_from_logits(s, t, "kl", teacher_flips=flags_dev),
                                                        s),
                            lambda: flip_eager(s, t, flags.tolist(), "kl"), 20 * C),
            }[wname]

        for wname in names:
            fw = [work(wname, *x) for x in sets]
            bpp = fw[0][2]
            ms_f = timed([graphed(f[0]) for f in fw], args.reps)
            ms_e = timed([f[1] for f in fw], max(args.reps // 4, 3))
            rate = bpp * npx / (ms_f * 1e-3)
            row = {"shape": name, "BCHW": [B, C, H, W], "loss": wname, "fused_ms": round(ms_f, 4),
                   "eager_ms": round(ms_e, 3), "speedup": round(ms_e / ms_f, 2), "fused_GBps": round(rate / 1e9, 1),
                   "share_of_peak": round(rate / peak, 3), "input_copies": ncopy}
            rows.append(row)
            print(f"{name:10s} ({B},{C},{H},{W}) {wname:10s} fused {ms_f:8.3f} ms  eager {ms_e:8.3f} ms  "
                  f"x{ms_e / ms_f:5.1f}  {rate / 1e12:5.2f} TB/s = {rate / peak:.3f} of peak")
        del sets
        torch.cuda.empty_cache()
    iic_b200.raise_if_flagged(dev)
    print(json.dumps({"card": card, "power_limit": power_limit(), "hbm_peak_TBps": round(peak / 1e12, 3),
                      "rows": rows}))


if __name__ == "__main__":
    main()
