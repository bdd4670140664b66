"""Times the global IIC terms from logits -- the finish launch normalising the (N, K) logit rows and
global_backward_kernel<true> -- against torch.softmax + the probability rows, in CUDA graphs: one iic_losses call of S
global terms (the Conv5 ClusterHead's sub-heads, views of one (2N, S*K) head output), forward + backward through
autograd.

    python tools/time_from_logits_global.py [--N 32] [--K 10] [--S 5] [--T 1.0]

Prints the GPU name and power limit with the numbers."""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import iic_b200  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_from_logits_k20 import graph_time  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, default=32, help="rows of one view (the per-GPU batch)")
    ap.add_argument("--K", type=int, default=10)
    ap.add_argument("--S", type=int, default=5, help="sub-heads: global terms in the call")
    ap.add_argument("--T", type=float, default=1.0)
    ap.add_argument("--reps", type=int, default=200)
    a = ap.parse_args()
    dev = torch.device("cuda:0")
    iic_b200.set_check_mode("deferred")
    try:
        plim = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        plim = "unknown"
    print(f"GPU {torch.cuda.get_device_name(dev)}, power limit {plim}; S = {a.S} global terms of ({a.N}, {a.K}), T {a.T}")
    gen = torch.Generator(device=dev).manual_seed(0)
    head = torch.randn(2 * a.N, a.S * a.K, device=dev, generator=gen).mul_(2).requires_grad_(True)
    crit = iic_b200.IIDLoss()

    def step(fused):
        def f():
            calls = []
            for s in range(a.S):
                x, y = torch.chunk(head[:, s * a.K:(s + 1) * a.K], 2, 0)
                if not fused:
                    x, y = (x / a.T).softmax(1), (y / a.T).softmax(1)
                calls.append((crit, x, y))
            out = iic_b200.iic_losses(calls, from_logits=fused, T=a.T)
            torch.autograd.grad(sum(o[0] for o in out), (head,))
        return f
    print(f"  {'iic_losses(from_logits=True) fwd+bwd':40s} {graph_time([step(True)], a.reps):9.1f} us")
    print(f"  {'softmax + iic_losses fwd+bwd':40s} {graph_time([step(False)], a.reps):9.1f} us")


if __name__ == "__main__":
    main()
