"""Times the softmax-fused local term (16 <= K <= 24, and K = 128 at padding 1) against torch.softmax + the probability
path, in CUDA graphs,
with inputs rotated over enough copies that the working set exceeds the 126 MB L2:

  forward   fused: stats pass + from-logits joint + finish     fallback: torch softmax x2 + joint + finish
  backward  fused: from-logits row-block backward               fallback: probability backward + softmax backward x2
  term      loss and logit gradients through autograd (IIDSegmentationSmallPathLoss.from_logits vs softmax + call)
  step      (--step) one S = 5 iic_losses(from_logits=True) call on the channel blocks of one (2B, S*K, H, W) head
            output, fwd + bwd, against softmax + iic_losses

    python tools/time_from_logits_k20.py --shape 8,20,224,224 --pad 3 [--T 1.0] [--step]
    python tools/time_from_logits_k20.py --shape 32,128,224,224 --pad 1        (the wide heads, BASELINE config 5)

Prints the GPU name and power limit with the numbers, and which path the fused side took (the coverage query)."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import iic_b200  # noqa: E402
from iic_b200 import ops as O  # noqa: E402

L2_BYTES = 126 << 20


def graph_time(fns, reps):
    """Mean time of one fn call (us): all fns captured in one CUDA graph, replayed `reps` times after a warm-up."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            for f in fns:
                f()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for f in fns:
            f()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        g.replay()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps / len(fns) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="8,20,224,224", help="B,K,H,W of one map")
    ap.add_argument("--K", type=int, default=None, help="override K of --shape")
    ap.add_argument("--pad", type=int, default=3)
    ap.add_argument("--T", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--step", action="store_true", help="also time one S = 5 iic_losses step")
    a = ap.parse_args()
    B, K, H, W = (int(v) for v in a.shape.split(","))
    K = a.K or K
    dev = torch.device("cuda:0")
    iic_b200.set_check_mode("deferred")
    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        plim = "unknown"
    print(f"GPU {torch.cuda.get_device_name(dev)}, power limit {plim}; shape ({B}, {K}, {H}, {W}) padding {a.pad} T {a.T}")
    inv_t = 1.0 / a.T
    map_bytes = B * K * H * W * 4
    nsets = max(1, -(-2 * L2_BYTES // (2 * map_bytes)))
    gen = torch.Generator(device=dev).manual_seed(0)
    sets = [(torch.randn(B, K, H, W, device=dev, generator=gen) * 2, torch.randn(B, K, H, W, device=dev, generator=gen) * 2)
            for _ in range(nsets)]
    covered = O.from_logits_covered(sets[0][0], sets[0][1], a.pad)
    print(f"fused path taken: {'yes' if covered else 'no (softmax + probability path)'}; {nsets} input sets "
          f"({nsets * 2 * map_bytes / 2**20:.0f} MiB)")
    one = torch.ones((), device=dev)
    res = {}

    # forward: joint + finish
    def fwd_fused(l1, l2):
        return lambda: O._finish_terms([O.LocalTerm(l1, l2, None, a.pad, (H, W), (H, W), 1.0, logits=True,
                                                    inv_temperature=inv_t)], False)

    def fwd_soft(l1, l2):
        return lambda: O._finish_terms([O.LocalTerm((l1 / a.T).softmax(1), (l2 / a.T).softmax(1), None, a.pad, (H, W),
                                                    (H, W), 1.0)], False)
    if covered:
        res["forward fused"] = graph_time([fwd_fused(*s) for s in sets], a.reps)
    res["forward softmax+prob"] = graph_time([fwd_soft(*s) for s in sets], a.reps)

    # backward (the forward's outputs computed once per set, outside the graph)
    gx = torch.empty(B, K, H, W, device=dev)
    gy = torch.empty(B, K, H, W, device=dev)
    if covered:
        recs = [fwd_fused(*s)()[0] for s in sets]
        res["backward fused"] = graph_time(
            [(lambda s=s, r=r: O._local_backward_logits_stats_into(s[0], s[1], r["stats"], r["Wx"], r["Wy"], one, a.pad,
                                                                   inv_t, gx, gy)) for s, r in zip(sets, recs)], a.reps)
        del recs
    probs = [((l1 / a.T).softmax(1), (l2 / a.T).softmax(1)) for l1, l2 in sets]
    precs = [O._finish_terms([O.LocalTerm(p1, p2, None, a.pad, (H, W), (H, W), 1.0)], False)[0] for p1, p2 in probs]

    def bwd_soft(p, r):
        def f():
            O._local_backward_into(p[0], p[1], None, r["Wx"], r["Wy"], one, a.pad, H, W, H, W, gx, gy)
            torch._softmax_backward_data(gx, p[0], 1, torch.float32).mul_(inv_t)
            torch._softmax_backward_data(gy, p[1], 1, torch.float32).mul_(inv_t)
        return f
    res["backward softmax+prob"] = graph_time([bwd_soft(p, r) for p, r in zip(probs, precs)], a.reps)
    del probs, precs

    # the whole term through autograd
    crit = iic_b200.IIDSegmentationSmallPathLoss(padding=a.pad, patch_size=4096)
    leaves = [(l1.requires_grad_(True), l2.requires_grad_(True)) for l1, l2 in sets]

    def term(l1, l2, fused):
        def f():
            loss = crit.from_logits(l1, l2, T=a.T) if fused else crit((l1 / a.T).softmax(1), (l2 / a.T).softmax(1))
            torch.autograd.grad(loss, (l1, l2))
        return f
    res["term fused" if covered else "term from_logits (fallback)"] = graph_time([term(*s, True) for s in leaves], a.reps)
    res["term softmax+prob"] = graph_time([term(*s, False) for s in leaves], a.reps)
    del leaves, sets

    if a.step:
        S = 5
        nst = max(1, -(-2 * L2_BYTES // (2 * S * map_bytes)))
        heads = [torch.randn(2 * B, S * K, H, W, device=dev, generator=gen).mul_(2).requires_grad_(True) for _ in range(nst)]

        def step(h, fused):
            def f():
                v = h.view(2 * B, S, K, H, W)
                calls = []
                for s in range(S):
                    x, y = torch.chunk(v[:, s], 2, 0)
                    if not fused:
                        x, y = (x / a.T).softmax(1), (y / a.T).softmax(1)
                    calls.append((crit, x, y))
                out = iic_b200.iic_losses(calls, from_logits=fused, T=a.T)
                torch.autograd.grad(sum(out), (h,))
            return f
        res[f"step S={S} iic_losses(from_logits=True)"] = graph_time([step(h, True) for h in heads], a.reps)
        res[f"step S={S} softmax + iic_losses"] = graph_time([step(h, False) for h in heads], a.reps)

    for k, v in res.items():
        print(f"  {k:40s} {v:9.1f} us")


if __name__ == "__main__":
    main()
