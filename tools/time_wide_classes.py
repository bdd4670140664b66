"""Times the wide-class (9 <= C <= 256) UDA, supervised and flip-aligned losses, forward + backward, against the
reference's formulas in eager torch on the same GPU.

    python tools/time_wide_classes.py [--reps N]

Fused: one CUDA graph per workload (forward and backward of the library's loss).  Eager: the reference's composition,
  UDA        softmax of both maps, then the KL_div expression (semi_seg/epocher.py:221-224; kl_losses.py:107-126)
             or torch.nn.MSELoss;
  supervised F.one_hot(long), the KL_div expression, logits.max(1)[1] and the one-hot Dice sums
             (epocher.py:165-166,183-184);
  flip       the per-sample flip loop and torch.stack (epocher.py:160-161), then the UDA term.
Every input map is larger than the 126 MB L2, so each pass streams from HBM.  Algorithmic bytes per pixel: 20*C for
UDA (forward reads 2C floats, backward reads 2C and writes C), 12*C + 16 for supervised (forward reads C floats and an
int64 label, backward reads the same and writes C).  The HBM peak is measured in the same run with a device-to-device
copy; the card's name and power limit are printed beside it.
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

SHAPES = [("cityscapes", (16, 19, 512, 1024)), ("voc", (16, 21, 512, 512)), ("ade", (8, 150, 256, 256))]
EPS = 1e-16


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


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
    ms = timed(lambda: dst.copy_(src), reps)
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
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_wide_classes.py needs a CUDA device")
    dev = torch.device("cuda:0")
    iic_b200.set_check_mode("deferred")
    card = torch.cuda.get_device_name(dev)
    peak = hbm_peak(dev, args.reps)
    print(f"card: {card}, power limit: {power_limit()}, measured HBM copy peak: {peak / 1e12:.2f} TB/s")
    rows = []
    for name, (B, C, H, W) in SHAPES:
        g = torch.Generator(device=dev).manual_seed(C)
        s = (torch.randn(B, C, H, W, device=dev, generator=g) * 2).requires_grad_(True)
        t = torch.randn(B, C, H, W, device=dev, generator=g) * 2
        lab = torch.randint(0, C, (B, H, W), device=dev, generator=g)
        flags = torch.arange(B, dtype=torch.uint8) % 4
        flags_dev = flags.to(dev)
        npx = B * H * W
        work = {
            "uda_kl": (lambda: torch.autograd.grad(iic_b200.uda_from_logits(s, t, "kl"), s),
                       lambda: uda_eager(s, t, "kl"), 20 * C),
            "uda_mse": (lambda: torch.autograd.grad(iic_b200.uda_from_logits(s, t, "mse"), s),
                        lambda: uda_eager(s, t, "mse"), 20 * C),
            "sup": (lambda: torch.autograd.grad(iic_b200.sup_kl_from_logits(s, lab, return_dice=True)[0], s),
                    lambda: sup_eager(s, lab, C), 12 * C + 16),
            "flip_kl": (lambda: torch.autograd.grad(iic_b200.uda_from_logits(s, t, "kl", teacher_flips=flags_dev), s),
                        lambda: flip_eager(s, t, flags.tolist(), "kl"), 20 * C),
        }
        for wname, (fused, eager, bpp) in work.items():
            ms_f = timed(graphed(fused), args.reps)
            ms_e = timed(eager, max(args.reps // 4, 3))
            rate = bpp * npx / (ms_f * 1e-3)
            row = {"shape": name, "BCHW": [B, C, H, W], "loss": wname, "fused_ms": round(ms_f, 4),
                   "eager_ms": round(ms_e, 3), "speedup": round(ms_e / ms_f, 2), "fused_GBps": round(rate / 1e9, 1),
                   "share_of_peak": round(rate / peak, 3)}
            rows.append(row)
            print(f"{name:10s} ({B},{C},{H},{W}) {wname:8s} fused {ms_f:8.3f} ms  eager {ms_e:8.3f} ms  "
                  f"x{ms_e / ms_f:5.1f}  {rate / 1e12:5.2f} TB/s = {rate / peak:.3f} of peak")
        del s, t, lab
        torch.cuda.empty_cache()
    iic_b200.raise_if_flagged(dev)
    print(json.dumps({"card": card, "power_limit": power_limit(), "hbm_peak_TBps": round(peak / 1e12, 3),
                      "rows": rows}))


if __name__ == "__main__":
    main()
