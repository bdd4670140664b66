"""Ill-conditioned inputs: near-uniform cluster maps (mutual information ~ 0, so J - min J cancels almost everything).

    python tools/near_uniform_check.py

Compares the tensor-core path, the FP32 path (the no_tc switch) and the fp64 oracle on the loss and the gradients for
K = 20 (padding 3) and K = 128 (padding 1) maps made by a weak random 1x1 head, the regime of the first training
iterations.
"""
import os, sys, torch, numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import iic_b200, iic_oracle as O
dev = torch.device("cuda:0")
torch.manual_seed(0)
for (B, K, H, W, pad, scale) in [(10, 20, 224, 224, 3, 0.05), (10, 20, 224, 224, 3, 0.5), (4, 20, 64, 64, 3, 0.05), (8, 128, 64, 64, 1, 0.05)]:
    f = torch.randn(B, 16, H, W, device=dev)
    w = torch.randn(K, 16, device=dev) * scale
    z1 = torch.einsum("kc,bchw->bkhw", w, f)
    z2 = torch.einsum("kc,bchw->bkhw", w, f + 0.3 * torch.randn_like(f))
    x = z1.softmax(1).contiguous().requires_grad_(True)
    y = z2.softmax(1).contiguous().requires_grad_(True)
    crit = iic_b200.IIDSegmentationSmallPathLoss(padding=pad, patch_size=1024)
    res = {}
    for mode in ("tc", "notc"):
        # the library reads IIC_B200_NO_TC once, when it loads: switch at run time
        iic_b200._lib.set_option("no_tc", 1 if mode == "notc" else 0)
        l = crit(x, y)
        gx, gy = torch.autograd.grad(l, (x, y))
        res[mode] = (l.item(), gx.clone(), gy.clone())
    ol = None
    if B * H * W <= 600000:
        ol, ogx, ogy = O.iid_segmentation_small_path_loss(x.detach().cpu().numpy(), y.detach().cpu().numpy(), pad, 1024, with_grads=True)
    lt, ln = res["tc"][0], res["notc"][0]
    gerr = (res["tc"][1] - res["notc"][1]).abs().max().item() / res["notc"][1].abs().max().item()
    print(f"B={B} K={K} {H}x{W} p={pad} scale={scale}: loss tc {lt:.8f} notc {ln:.8f} rel diff {abs(lt-ln)/abs(ln):.2e}  grad tc-vs-notc {gerr:.2e}  oracle {ol}")
    if ol is not None:
        print(f"    vs oracle: tc {abs(lt-ol)/abs(ol):.2e}  notc {abs(ln-ol)/abs(ol):.2e}; grad tc {np.abs(res['tc'][1].cpu().numpy()-ogx).max()/np.abs(ogx).max():.2e} notc {np.abs(res['notc'][1].cpu().numpy()-ogx).max()/np.abs(ogx).max():.2e}")
