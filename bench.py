#!/usr/bin/env python
"""Benchmark of the IIC MI loss hot path (BASELINE.json: "IIC MI loss fwd+bwd Mpixels/s").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 2|3|4|5] [--workload udaiic]
                    [--dump-outputs DIR]

Headline workload at every N (weak scaling, per-GPU work fixed) = BASELINE config 2: global + local IIC (padding 1,
patch 512, i.e. one patch) on Up_conv2-shaped maps, per GPU 32 x 10 x 224 x 224 float32 probability maps for the two
views plus the (32, 10) global head, forward + backward to both inputs.  One "step" = local small-patch loss + global
IIDLoss, summed, backward -- evaluated through the public batched call ``iic_b200.iic_losses`` (one joint kernel, ONE
finish launch for both terms incl. the multi-GPU exchange, two backward kernels).  A pixel = one (n, u, v) site of one
loss call (SURVEY.md 8d).  ``--config 3|4|5`` select the other BASELINE configurations as whole workloads.

The JSON line carries, beyond the base contract:
  value     device-timed throughput, inputs resident in HBM (CUDA-graph replay of the public-API step)
  e2e       the same through the public modules with HOST (pinned, NUMA-local) inputs: H2D of every input, forward,
            backward, D2H of the loss, every step; e2e.with_gradients adds the D2H of every input gradient
  roofline  the dominant kernel (the local backward; one launch per step at config 2): algorithmic bytes per launch
            (16*K bytes/px: read both K-channel maps, write both gradients) over its CUDA-event duration, against
            MEASURED_PEAKS.json's HBM copy bandwidth
  cpu_baseline  the reference's own loss classes (oracle/_ref, loaded by oracle/ref_loader.py) on the host cores
  extra     secondary shapes and terms, and the whole udaiic iteration on the reference's own epocher
  dumped_outputs  with ``--dump-outputs DIR``: which arrays were written there

``--impl reference`` times the reference's own CPU implementation of the same workload (same config dict).

``--dump-outputs DIR`` writes what the last of the ``--steps`` timed steps returned -- the total loss and the gradient of
every differentiable input -- as ``DIR/<name>.npy`` (float32, at most 60 MiB in all; a large gradient is stored as a fixed,
seeded sample of its elements).  The inputs depend only on the arguments, so two builds can be compared array by array;
the local-term gradients vary by a few float32 ulps from run to run (the order of their reductions is not fixed), so
compare them with a tolerance.
"""
from __future__ import annotations

import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "iic_mi_loss_fwd_bwd_mpixels_per_s"
UNIT = "Mpx/s"
NSETS = 4          # rotating input sets

# ---------------------------------------------------------------------------------------------------------------------
# workloads: groups of IIC terms.  group = (kind, S sub-heads, K, H, W, padding, patch_size, weight)
# total = sum_g weight_g * mean_s L_gs  (+ uda_weight * UDA): config 2 is "local + global", config 3 the udaiic
# regulariser with the yaml weights (semi.yaml:31-61: importance [1, .5, .5] normalised, iic 0.1, uda mse 5.0)
# ---------------------------------------------------------------------------------------------------------------------
WORKLOADS = {
    2: dict(name="config2: global+local IIC (padding=1, patch 512) on Up_conv2-shaped maps, batch 32 fp32 per GPU, fwd+bwd",
            batch_per_gpu=32, batch_total=None, scaling="weak",
            groups=[("local", 1, 10, 224, 224, 1, 512, 1.0), ("global", 1, 10, 0, 0, 0, 0, 1.0)], uda=None),
    3: dict(name="config3: multi-head IIC (5 sub-heads x {Conv5 global, Up_conv3 p=1, Up_conv2 p=3}, K=20) + UDA mse, "
                 "8 samples per GPU (batch 64 over 8 GPUs), fwd+bwd",
            batch_per_gpu=8, batch_total=None, scaling="weak",
            groups=[("global", 5, 20, 0, 0, 0, 0, 0.1 * 0.5), ("local", 5, 20, 112, 112, 1, 1024, 0.1 * 0.25),
                    ("local", 5, 20, 224, 224, 3, 1024, 0.1 * 0.25)], uda=(4, 224, 224, 5.0)),
    4: dict(name="config4: high-res 512x512, 20 clusters, local MI padding=3, batch 128 over the GPUs, fwd+bwd",
            batch_per_gpu=None, batch_total=128, scaling="strong",
            groups=[("local", 1, 20, 512, 512, 3, 1024, 1.0)], uda=None),
    5: dict(name="config5: wide-cluster K=128 global+local IIC (padding=1, tensor-core contraction), 32 samples per GPU "
                 "(batch 256 over 8 GPUs), fwd+bwd",
            batch_per_gpu=32, batch_total=None, scaling="weak",
            groups=[("local", 1, 128, 224, 224, 1, 512, 1.0), ("global", 1, 128, 0, 0, 0, 0, 1.0)], uda=None),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(WORKLOADS))
    ap.add_argument("--workload", default="loss", choices=["loss", "udaiic"],
                    help="udaiic: whole training iterations/s of the reference's UDAIICEpocher, losses swapped vs not")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and input gradients of the last timed step as DIR/<name>.npy (float32; "
                         "rank 0's shard when several GPUs run)")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 2000 if (a.config == 2 and a.impl == "b200") else 20
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload != "loss"):
        ap.error("--dump-outputs applies to the loss workload of the b200 implementation")
    return a


def batch_of(wl, world):
    return wl["batch_per_gpu"] if wl["batch_per_gpu"] else max(wl["batch_total"] // world, 1)


def pixels_per_step(wl, B):
    return sum(S * B * (H * W if kind == "local" else 1) for kind, S, K, H, W, pad, patch, w in wl["groups"])


def input_set_bytes(wl, B):
    b = sum(2 * 4 * S * K * B * (H * W if kind == "local" else 1) for kind, S, K, H, W, pad, patch, w in wl["groups"])
    if wl["uda"]:
        b += 2 * 4 * B * wl["uda"][0] * wl["uda"][1] * wl["uda"][2]
    return b


def workload_config(cfg_id, world):
    """The `config` object of the JSON line -- identical for both arms."""
    wl = WORKLOADS[cfg_id]
    B = batch_of(wl, world)
    return {"workload": wl["name"], "config_id": cfg_id, "B_per_gpu": B,
            "terms": [{"kind": k, "sub_heads": S, "K": K, "H": H, "W": W, "padding": pad, "patch_size": patch}
                      for k, S, K, H, W, pad, patch, w in wl["groups"]],
            "uda": None if not wl["uda"] else {"C": wl["uda"][0], "H": wl["uda"][1], "W": wl["uda"][2], "kind": "mse"},
            "pixels_per_step_per_gpu": pixels_per_step(wl, B),
            "l2": f"inputs rotate over {NSETS} sets of {input_set_bytes(wl, B) / 1e6:.0f} MB "
                  f"({NSETS * input_set_bytes(wl, B) / 1e6:.0f} MB in flight, L2 is 126 MB)"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)", float(d.get("sm_max_mhz", 1965.0)), \
            float(d.get("bf16_tflops", 1590.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0, 1590.0


# dram bytes per launch of the dominant kernel from one `ncu --set full` capture; None until measured for the current kernel
TRAFFIC_BWD = (211.2e6, "ncu --set full, profiles/r02_ncu_config2_kernels_tcjoint.txt (local_bwd_tcrb10h_kernel): dram__bytes_read 133.3 MB + "
               "dram__bytes_write 77.9 MB per launch (algorithmic 256.9 MB; the tail of the gradient writes is still in L2)")


# ---------------------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY 8d: correlated views so MI is O(0.1-1)); per group one (B, S*K, ...) tensor per view whose
# S channel blocks are the sub-heads, exactly what the batched cluster heads emit (softmax per sub-head)
# ---------------------------------------------------------------------------------------------------------------------
def make_inputs(torch, device, seed, wl, B):
    g = torch.Generator(device=device).manual_seed(seed)
    tensors = []
    for kind, S, K, H, W, pad, patch, w in wl["groups"]:
        if kind == "local":
            base = torch.randn(B, S * K, max(H // 8, 1), max(W // 8, 1), device=device, generator=g) * 3
            base = torch.nn.functional.interpolate(base, size=(H, W), mode="bilinear", align_corners=False)
            for _ in range(2):
                l = base + 0.5 * torch.randn(B, S * K, H, W, device=device, generator=g)
                tensors.append(l.view(B, S, K, H, W).softmax(2).view(B, S * K, H, W).contiguous())
                del l
            del base
        else:
            gb = torch.randn(B, S * K, device=device, generator=g) * 2
            for _ in range(2):
                l = gb + 0.7 * torch.randn(B, S * K, device=device, generator=g)
                tensors.append(l.view(B, S, K).softmax(2).view(B, S * K).contiguous())
    if wl["uda"]:
        C, H, W, _ = wl["uda"]
        tensors.append(torch.randn(B, C, H, W, device=device, generator=g) * 2)      # student logits (gets the gradient)
        tensors.append(torch.randn(B, C, H, W, device=device, generator=g) * 2)      # teacher logits
    return tensors


def grad_mask(wl):
    """Which input tensors receive a gradient (the UDA teacher does not)."""
    m = [True] * (2 * len(wl["groups"]))
    if wl["uda"]:
        m += [True, False]
    return m


def build_step(wl, B, crits, iic_losses, uda_fn, torch):
    """step(tensors) -> (total loss, gradients of every differentiable input) through the given loss callables."""

    def step(tensors):
        calls, spans = [], []
        for gi, (kind, S, K, H, W, pad, patch, w) in enumerate(wl["groups"]):
            x, y = tensors[2 * gi], tensors[2 * gi + 1]
            spans.append((len(calls), S, w))
            if S == 1:
                calls.append((crits[gi], x, y))
                continue
            # the S sub-heads are channel blocks of ONE head output, as the batched cluster heads emit them
            if kind == "local":
                xv, yv = x.view(B, S, K, H, W), y.view(B, S, K, H, W)
            else:
                xv, yv = x.view(B, S, K), y.view(B, S, K)
            calls += [(crits[gi], xv[:, s], yv[:, s]) for s in range(S)]
        losses = iic_losses(calls)
        flat = [l[0] if isinstance(l, tuple) else l for l in losses]
        total = None
        for start, S, w in spans:
            part = flat[start] if S == 1 else torch.stack(flat[start:start + S]).mean()
            part = part if w == 1.0 else part * w
            total = part if total is None else total + part
        if wl["uda"]:
            total = total + wl["uda"][3] * uda_fn(tensors[-2], tensors[-1])
        diff = [t for t, m in zip(tensors, grad_mask(wl)) if m]
        return total, torch.autograd.grad(total, diff)

    return step


DUMP_BYTES = 60 * 2**20        # --dump-outputs writes at most this many bytes of array data


def output_names(wl):
    """Names of what build_step's step returns: the total loss, then the gradient of every differentiable input."""
    names = ["loss"]
    for gi, (kind, *_rest) in enumerate(wl["groups"]):
        names += [f"grad_{gi}_{kind}_x", f"grad_{gi}_{kind}_y"]
    if wl["uda"]:
        names.append("grad_uda_student")
    return names


def dump_outputs(out_dir, wl, loss, grads, seed=0):
    """Writes the loss and the gradients of one step as out_dir/<name>.npy in float32, DUMP_BYTES in all.  The arrays
    are taken smallest first, each with an equal share of what the ones before it left unused; an array larger than its
    share is replaced by the elements at a fixed, seeded set of flat indices (sorted), the same set for the same shapes,
    so that two builds of the project can be compared output for output."""
    import numpy as np
    arrays = [loss.detach().reshape(1)] + [g.detach() for g in grads]
    names = output_names(wl)
    assert len(names) == len(arrays), (names, len(arrays))
    left = DUMP_BYTES // 4
    os.makedirs(out_dir, exist_ok=True)
    written = {}
    for n, i in enumerate(sorted(range(len(arrays)), key=lambda i: arrays[i].numel())):
        t = arrays[i]
        a = t.float().cpu().numpy().reshape(-1)
        cap = left // (len(arrays) - n)
        if a.size > cap:
            idx = np.random.default_rng([seed, a.size, cap]).choice(a.size, size=cap, replace=False)
            a = a[np.sort(idx)]
        left -= a.size
        np.save(os.path.join(out_dir, names[i] + ".npy"), np.ascontiguousarray(a, dtype=np.float32))
        written[names[i]] = {"numel": int(t.numel()), "written": int(a.size)}
    return {name: written[name] for name in names}


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the reference's own loss classes on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def load_reference_losses():
    """(namespace, kind): the UNMODIFIED reference classes (oracle/ref_loader.py: /root/reference here, the oracle/_ref
    copy on the GPU box) -> "reference"; the operator-for-operator port of oracle/torch_port.py -> "port" when absent."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_loader
        if ref_loader.available():
            with contextlib.redirect_stdout(sys.stderr):
                return ref_loader.load(), "reference"
    except Exception as e:  # noqa: BLE001
        print(f"[bench] reference classes unavailable ({type(e).__name__}: {e}); using oracle/torch_port.py", file=sys.stderr)
    import torch_port as TP
    return TP, "port"


def cpu_reference_run(cfg_id, world, steps, warmup, budget_s=150.0):
    """Times the reference's CPU implementation of the workload.  Returns dict(value, ms, threads, kind, batch, sample)."""
    import torch
    wl = WORKLOADS[cfg_id]
    ns, kind = load_reference_losses()
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    B_full = batch_of(wl, world)
    dev = torch.device("cpu")

    def crit_for(group):
        k, S, K, H, W, pad, patch, w = group
        with contextlib.redirect_stdout(sys.stderr):
            if kind == "reference":
                return ns.IIDSegmentationSmallPathLoss(padding=pad, patch_size=patch) if k == "local" else ns.IIDLoss()
            if k == "local":
                return lambda a, b, _p=pad, _s=patch: ns.iid_segmentation_small_path_loss(a, b, _p, _s)
            return lambda a, b: ns.iid_loss(a, b)

    crits = [crit_for(g) for g in wl["groups"]]

    def ref_losses(calls):
        out = []
        for c, a, b in calls:
            # the epocher feeds chunk() halves of a head output: contiguous per-head maps, leaves of the graph here
            r = c(a.contiguous(), b.contiguous())
            out.append(r[0] if isinstance(r, tuple) else r)
        return out

    def uda(a, b):            # semi_seg/epocher.py:221-224 with nn.MSELoss (trainer.py:194)
        return torch.nn.functional.mse_loss(a.softmax(1), b.softmax(1).detach())

    def run(B, n_steps, n_warm, nsets):
        step = build_step(wl, B, crits, ref_losses, uda, torch)
        sets = [[t.requires_grad_(m) for t, m in zip(make_inputs(torch, dev, 1236 + 17 * s, wl, B), grad_mask(wl))]
                for s in range(nsets)]
        for i in range(n_warm):
            step(sets[i % nsets])
        times = []
        for i in range(n_steps):
            t0 = time.perf_counter()
            loss, _ = step(sets[i % nsets])
            float(loss.detach())
            times.append(time.perf_counter() - t0)
        return times

    # size the per-step sample so that the whole run ends within `budget_s`: grow the batch from 1 by doubling while the
    # MEASURED step time says the run still fits (CPU time is far from linear in the batch for the large-filter conv2d)
    B, t_last = 1, None
    while True:
        t_last = min(run(B, 1, 0 if t_last is not None else 1, 1))
        nxt = min(2 * B, B_full)
        if B == B_full or 2.2 * t_last * (nxt / B) / 2.0 * (steps + warmup) > budget_s:
            break
        B = nxt
    if t_last * (steps + warmup) > 3 * budget_s and B > 1:
        B //= 2
    nsets = NSETS if NSETS * input_set_bytes(wl, B) < 8e9 else 1
    times = run(B, steps, warmup, nsets)
    ms = statistics.mean(times) * 1e3
    px = pixels_per_step(wl, B)
    sample = (f"{'full' if B == B_full else 'bounded'} sample: batch {B} of {B_full} per step, "
              f"mean of {steps} timed steps after {warmup} warm-up, {threads} threads, "
              + ("the reference's own IIDSegmentationSmallPathLoss / IIDLoss (unmodified, oracle/ref_loader.py)"
                 if kind == "reference" else "oracle/torch_port.py (operator-for-operator port; reference copy absent)"))
    return {"value": px / (ms * 1e-3) / 1e6, "ms": ms, "best_ms": min(times) * 1e3, "threads": threads, "kind": kind, "batch": B,
            "batch_full": B_full, "sample": sample}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    r = cpu_reference_run(args.config, world, max(args.steps, 1), max(args.warmup, 0))
    cfg = workload_config(args.config, world)
    line = {"impl": "reference", "metric": METRIC, "value": round(r["value"], 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(r["ms"], 3), "higher_is_better": True,
            "scaling": WORKLOADS[args.config]["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": round(r["value"], 4), "unit": UNIT, "cores": r["threads"], "kind": r["kind"],
                             "sample": r["sample"]},
            "e2e": {"value": round(r["value"], 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "one process on the host cores of the box (rank 0 only); value = pixels of ONE rank's step / time, "
                    "i.e. the CPU path does not scale with --gpus"}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# helpers of the B200 arm
# ---------------------------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local_rank):
    """Pin this process (and therefore the first touch of its pinned buffers) to the NUMA node of its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"node": None, "note": "the platform reports no NUMA affinity for the GPU"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"node": node, "cpus_bound": len(allowed)}
    except Exception as e:  # noqa: BLE001
        return {"node": None, "note": f"not bound ({type(e).__name__}: {e})"}


def count_own_launches(torch, fn):
    """Kernels of libiic_b200.so launched by one eager call of `fn` (all of them live in namespace iic::)."""
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        names = [e.name for e in prof.events() if getattr(e, "device_type", None) is not None and "iic::" in e.name]
        own = [n for n in names if "iic::" in n]
        return len(own), sorted(set(n.split("(")[0].split("<")[0] for n in own))
    except Exception as e:  # noqa: BLE001
        return None, [f"profiler unavailable: {type(e).__name__}"]


def static_launch_count(wl, world):
    """Fallback for gpu_launches when the profiler is unavailable: kernels of libiic_b200.so per step, from the dispatch
    rules (joint 1; finish 1 + 1 batched epilogue launch, +1 rank sum when a large batch is exchanged; backward 1 per
    local term, or 2 sweeps + 2 weight images on the K = 20 / K = 128 tensor-core kernels; global backward 1; UDA 2)."""
    n, units, entries = 0, 0, 0
    for kind, S, K, H, W, pad, patch, w in wl["groups"]:
        T2 = (2 * pad + 1) ** 2
        if kind == "local":
            n += S * (1 + (1 if K <= 10 else 4))
            units += S * T2
            entries += S * T2 * K * K
        else:
            n += S
            units += S
            entries += S * K * K
    big = units > 32 or entries > 1056
    n += 2 + (1 if (big and world > 1) else 0)
    if wl["uda"]:
        n += 2
    return n


def udaiic_iteration_extra(dev, iters=8):
    """Whole udaiic training iterations/s on the REFERENCE's own UDAIICEpocher (semi_seg/epocher.py:137-188,308-323,
    loaded unmodified from oracle/_ref by oracle/ref_epocher.py), yaml defaults (K = 20, 5 sub-heads, layers Conv5 /
    Up_conv3 / Up_conv2, paddings [1, 3], mse UDA), labeled 4 + unlabeled 4 at 224^2, synthetic device batches:
    INTEGRATION.md's three import swaps applied ("b200") vs not ("reference": the reference's torch losses on the
    same GPU).  The reference harness calls the product here, not the other way round."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_epocher as RE
    import iic_b200
    out = {"what": "reference UDAIICEpocher.run() (unmodified, oracle/_ref) over synthetic device batches, yaml defaults "
                   "K=20 S=5 layers Conv5/Up_conv3/Up_conv2 paddings [1,3] mse UDA, labeled 4 + unlabeled 4, 224x224; "
                   "loss classes swapped per INTEGRATION.md section 2 vs the reference's own torch losses on the same GPU"}
    tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    for arm in ("reference", "b200", "b200_deferred_checks"):
        prev = iic_b200.get_check_mode()
        try:
            torch.backends.cudnn.allow_tf32 = False              # the reference's conv2d-as-joint must not run in TF32
            torch.backends.cuda.matmul.allow_tf32 = False
            if arm == "b200_deferred_checks":                    # INTEGRATION.md's optional line: asserts stay on the device,
                iic_b200.set_check_mode("deferred")              # read once per epoch here
            swap = "reference" if arm == "reference" else "b200"
            ep, _, _ = RE.build_epocher(RE.YAML_DEFAULT, dev, labeled_bs=4, unlabeled_bs=4, num_batches=2, swap=swap)
            RE.run_epoch(ep)                                     # warm-up epoch (cuDNN autotune, allocator)
            ep, _, _ = RE.build_epocher(RE.YAML_DEFAULT, dev, labeled_bs=4, unlabeled_bs=4, num_batches=iters, swap=swap)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = RE.run_epoch(ep)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if arm != "reference":
                iic_b200.raise_if_flagged(torch.device(dev))
            try:
                reg = float(res["reg_loss"]["mean"])
            except Exception:  # noqa: BLE001
                reg = None
            out[arm] = {"it_per_s": round(iters / dt, 2), "ms_per_it": round(dt / iters * 1e3, 2), "reg_loss_mean": reg}
        except Exception as e:  # noqa: BLE001
            out[arm] = {"error": f"{type(e).__name__}: {e}"}
        finally:
            iic_b200.set_check_mode(prev)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    if "it_per_s" in out.get("reference", {}) and "it_per_s" in out.get("b200", {}):
        out["speedup"] = round(out["b200"]["it_per_s"] / out["reference"]["it_per_s"], 2)
    return out


# ---------------------------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import iic_b200
    from iic_b200 import ops as iops

    if args.workload == "udaiic":
        if rank == 0:
            print(json.dumps({"metric": "udaiic_training_iterations_per_s", "unit": "it/s", "n_gpus": 1,
                              "higher_is_better": True, "data": "synthetic", "result": udaiic_iteration_extra(dev, max(args.steps, 4))}))
        return

    iic_b200.set_check_mode("deferred")       # checks run on the device; flags are read after the timed region
    iic_b200.set_data_parallel(world > 1)
    wl = WORKLOADS[args.config]
    B = batch_of(wl, world)
    hbm_peak, peak_src, sm_max, bf16_peak = peaks()
    px_step = pixels_per_step(wl, B)
    px_job = px_step * world

    with contextlib.redirect_stdout(sys.stderr):      # the constructors print "Initialize ..." like the reference's
        crits = [iic_b200.IIDSegmentationSmallPathLoss(padding=pad, patch_size=patch) if kind == "local" else iic_b200.IIDLoss()
                 for kind, S, K, H, W, pad, patch, w in wl["groups"]]
    uda_fn = lambda a, b: iic_b200.uda_from_logits(a, b, "mse")      # noqa: E731
    step_fn = build_step(wl, B, crits, iic_b200.iic_losses, uda_fn, torch)

    # rotating input sets so every step's inputs come from HBM, not from L2
    sets = []
    for s in range(NSETS):
        ts = make_inputs(torch, dev, 1236 + 17 * s + 1000 * rank, wl, B)
        sets.append([t.requires_grad_(m) for t, m in zip(ts, grad_mask(wl))])
    set_bytes = sum(t.numel() * 4 for t in sets[0])

    # ---- CUDA graphs of the public-API step (one per input set) ----
    graphs, use_graph = [], not args.no_graph
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for inp in sets:
            for _ in range(2):
                out = step_fn(inp)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    n_own, own_names = count_own_launches(torch, lambda: step_fn(sets[0]))      # on EVERY rank: the step holds an exchange
    if use_graph:
        try:
            for inp in sets:
                gph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(gph, stream=side):
                    out = step_fn(inp)
                graphs.append((gph, out))
        except Exception as e:  # noqa: BLE001
            if rank == 0:
                print(f"[bench] CUDA graph capture failed ({type(e).__name__}: {e}); timing eager launches", file=sys.stderr)
            graphs, use_graph = [], False
            torch.cuda.synchronize()

    def run_one(i):
        """One step on input set i % NSETS; returns its (loss, gradients)."""
        if use_graph:
            graphs[i % NSETS][0].replay()
            return graphs[i % NSETS][1]
        return step_fn(sets[i % NSETS])

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    for i in range(max(args.warmup, 3)):
        run_one(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.perf_counter()
    e0.record()
    for i in range(args.steps):
        last = run_one(i)
    e1.record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps
    value = px_job / (ms_step * 1e-3) / 1e6
    iic_b200.raise_if_flagged(dev)           # the deferred simplex / NaN checks of every step above
    dumped = dump_outputs(args.dump_outputs, wl, *last) if (args.dump_outputs and rank == 0) else None
    del last

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731

    def timed_graph(fn, reps=20):
        """One op captured alone in a CUDA graph and replayed: device time only, CUDA events on the replay stream."""
        side2 = torch.cuda.Stream(device=dev)
        side2.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side2):
            for _ in range(2):
                fn()
        torch.cuda.current_stream().wait_stream(side2)
        torch.cuda.synchronize()
        g_ = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_, stream=side2):
            fn()
        for _ in range(3):
            g_.replay()
        torch.cuda.synchronize()
        t0, t1 = ev(), ev()
        t0.record()
        for _ in range(reps):
            g_.replay()
        t1.record()
        torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / reps
        del g_
        return ms

    # ---- multi-GPU correctness of the very step that was timed (outside the timed region) ----
    mg = None
    if world > 1:
        with torch.no_grad():
            pass
        wl_iic = dict(wl, uda=None)                  # the UDA term is a per-rank mean: only the IIC terms are exchanged
        n_iic = 2 * len(wl["groups"])
        loss_dp, grads_dp = build_step(wl_iic, B, crits, iic_b200.iic_losses, uda_fn, torch)(sets[0][:n_iic])
        bits = loss_dp.detach().view(torch.int32).clone()
        allbits = [torch.zeros_like(bits) for _ in range(world)]
        dist.all_gather(allbits, bits)
        identical = all(int(b.item()) == int(allbits[0].item()) for b in allbits)
        # rank 0 recomputes the loss of the concatenated batch on ONE GPU (exchange off) and compares
        gathered = []
        for t_ in sets[0][:n_iic]:
            buf = [torch.empty_like(t_) for _ in range(world)] if rank == 0 else None
            dist.gather(t_.detach(), buf, dst=0)
            gathered.append(torch.cat(buf, 0).requires_grad_(t_.requires_grad) if rank == 0 else None)
        mg = {"loss_bits_identical_on_all_ranks": bool(identical)}
        if rank == 0:
            iops._dist_enabled = False               # this rank only, and only for this call: no collective teardown
            try:
                full_step = build_step(wl_iic, B * world, crits, iic_b200.iic_losses, uda_fn, torch)
                loss_full, grads_full = full_step(gathered)
            finally:
                iops._dist_enabled = True
            rel = abs(loss_full.item() - loss_dp.item()) / max(abs(loss_full.item()), 1e-12)
            gd = grads_dp[0].double()
            gf = grads_full[0][:B].double()
            grel = float((gd - gf).abs().max() / gf.abs().max())
            mg.update({"loss_rel_diff_vs_one_gpu_on_concatenated_batch": rel, "shard_grad_rel_diff": grel,
                       "ok": bool(identical and rel <= 2e-6 and grel <= 1e-4)})
            del gathered, loss_full, grads_full
        dist.barrier(device_ids=[local_rank])
        iic_b200.set_check_mode("deferred")

    # ---- per-kernel timing of the dominant local term ----
    roofline, extra = None, {}
    gi_dom = max((i for i, g in enumerate(wl["groups"]) if g[0] == "local"), key=lambda i: wl["groups"][i][3] * wl["groups"][i][4] * wl["groups"][i][2])
    kind, S, K, H, W, pad, patch, w = wl["groups"][gi_dom]
    xs = sets[0][2 * gi_dom].detach().view(B, S, K, H, W)[:, 0]
    ys = sets[0][2 * gi_dom + 1].detach().view(B, S, K, H, W)[:, 0]
    one = torch.ones((), device=dev)
    half = patch // 2
    saved_dp = iops._dist_enabled
    iops._dist_enabled = False                      # single-op timings: no exchange
    try:
        J0 = iops.ops.local_joint(xs, ys, None, pad, patch, patch, half, half, True)
        _, Wx0, Wy0 = iops.ops.local_epilogue(J0, K, pad, 1.0)
        t_joint = timed_graph(lambda: iops.ops.local_joint(xs, ys, None, pad, patch, patch, half, half, True))
        t_epi = timed_graph(lambda: iops.ops.local_epilogue(J0, K, pad, 1.0))
        t_bwd = timed_graph(lambda: iops.ops.local_backward(xs, ys, None, Wx0, Wy0, one, pad, patch, patch, half, half))
        xr, yr = xs.clone().requires_grad_(True), ys.clone().requires_grad_(True)
        t_fwd = timed_graph(lambda: crits[gi_dom](xr, yr))            # joint + finish launch + epilogue launch
    finally:
        iops._dist_enabled = saved_dp
    alg_bytes_launch = 16.0 * K * B * H * W                   # read both maps + write both gradients, fp32
    achieved = alg_bytes_launch / (t_bwd * 1e-3) / 1e9
    sm_mhz = (clocks or {}).get("sm_mhz") or sm_max
    T2 = (2 * pad + 1) ** 2
    fma_per_launch = 2 * K * K * T2 * B * H * W               # useful FMAs of both sweeps
    fp32_peak = 148 * 128 * sm_mhz * 1e6                      # FMA/s at the observed clock
    tc10 = (K in (9, 10) and pad == 1 and not iic_b200._lib.load().iic_b200_get_option(b"no_tc")
            and not iic_b200._lib.load().iic_b200_get_option(b"no_tc10"))
    if K in (9, 10) and pad == 1:
        kname = ("local_bwd_tcrb10h_kernel (tcgen05 kind::f16 on fp16-split operands, both gradient sweeps in one launch)" if tc10
                 else "local_bwd_fast_kernel<10,1,16,4,5,false>")
    elif 16 <= K <= 24:
        kname = "local_bwd_tcrb_kernel (tcgen05 row-block sweeps, one launch per gradient + weight images)"
    elif K == 128:
        kname = "local_bwd_tc_kernel (tcgen05, one launch per gradient + weight images)"
    else:
        kname = "local backward"
    roofline = {"kernel": kname, "bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                "frac": round(achieved / hbm_peak, 4),
                "traffic": TRAFFIC_BWD[0] if (tc10 and args.config == 2) else None,
                "traffic_source": TRAFFIC_BWD[1] if (tc10 and args.config == 2) else None,
                "peak_source": peak_src, "launch_ms": round(t_bwd, 4),
                "algorithmic_bytes_per_launch": alg_bytes_launch,
                "note": "the local backward of the largest term, timed alone (single-op CUDA graph, CUDA events); it runs on the "
                        "tensor cores (fp32-accurate split products) and is bound by its MMA stream (12 MMAs per source row), not by HBM; "
                        "fp32_fma_frac compares its useful FMAs with the FP32 SIMT peak it replaced",
                "fp32_fma_frac": round(fma_per_launch / (t_bwd * 1e-3) / fp32_peak, 4),
                "step_breakdown_ms": {"local_joint+separate_reduce(+simplex)": round(t_joint, 4),
                                      "local_epilogue_separate": round(t_epi, 4),
                                      "local_forward_joint+finish (what the step runs)": round(t_fwd, 4),
                                      "local_backward": round(t_bwd, 4)},
                "whole_step_hbm_frac": round(24.0 * sum(S_ * K_ * B * (H_ * W_ if k_ == "local" else 1)
                                                         for k_, S_, K_, H_, W_, p_, ps_, w_ in wl["groups"])
                                             / (ms_step * 1e-3) / 1e9 / hbm_peak, 4)}

    # ---- secondary lines (config 2 only; not the headline) ----
    if args.config == 2 and not args.no_extra:
        local = crits[0]
        try:
            gl = torch.Generator(device=dev).manual_seed(99 + rank)
            lbase = torch.nn.functional.interpolate(torch.randn(B, K, H // 8, W // 8, device=dev, generator=gl) * 3,
                                                    size=(H, W), mode="bilinear", align_corners=False)
            l1 = (lbase + 0.5 * torch.randn(B, K, H, W, device=dev, generator=gl)).requires_grad_(True)
            l2 = (lbase + 0.5 * torch.randn(B, K, H, W, device=dev, generator=gl)).requires_grad_(True)
            ms_fused = timed_graph(lambda: torch.autograd.grad(local.from_logits(l1, l2), (l1, l2)))
            ms_unfused = timed_graph(lambda: torch.autograd.grad(local(l1.softmax(1), l2.softmax(1)), (l1, l2)))
            extra["local_from_logits"] = {
                "what": "local IIC fwd+bwd from the cluster head's LOGITS (softmax fused into the kernels) vs "
                        "torch softmax + the probability kernels + torch softmax backward, same shape",
                "fused_ms": round(ms_fused, 4), "torch_softmax_plus_probs_ms": round(ms_unfused, 4),
                "fused_mpx_s": round(B * H * W / (ms_fused * 1e-3) / 1e6, 1)}
            C_ = 4
            u1 = (torch.randn(B, C_, H, W, device=dev, generator=gl) * 2).requires_grad_(True)
            u2 = torch.randn(B, C_, H, W, device=dev, generator=gl) * 2
            ms_uda = timed_graph(lambda: torch.autograd.grad(iic_b200.uda_from_logits(u1, u2, "mse"), (u1,)))
            uda_bytes = 20.0 * C_ * B * H * W
            extra["uda_mse_from_logits"] = {
                "what": "UDA consistency fwd+bwd, (B,4,H,W), softmax fused; algorithmic bytes 20*C per pixel",
                "ms": round(ms_uda, 4), "gb_s": round(uda_bytes / (ms_uda * 1e-3) / 1e9, 1),
                "hbm_frac": round(uda_bytes / (ms_uda * 1e-3) / 1e9 / hbm_peak, 4),
                "note": "32 MB working set: L2-resident between replays, so this is an upper bound on HBM efficiency"}
            del l1, l2, lbase, u1, u2
        except Exception as e:  # noqa: BLE001
            extra["error"] = f"{type(e).__name__}: {e}"
        try:
            # streaming kernels of SURVEY 8f with inputs rotating over 4 sets inside one graph replay (> 126 MB L2): from HBM
            NR = 4
            gr = torch.Generator(device=dev).manual_seed(399 + rank)
            rs = [(torch.randn(B, 4, H, W, device=dev, generator=gr) * 2).requires_grad_(True) for _ in range(NR)]
            rt = [torch.randn(B, 4, H, W, device=dev, generator=gr) * 2 for _ in range(NR)]
            rl = [torch.randint(0, 4, (B, H, W), device=dev, generator=gr) for _ in range(NR)]
            rf = iic_b200.draw_flip_flags(4321, B).to(dev)
            fl = [int(v) for v in rf.tolist()]

            def sup_rot():
                for a_, l_ in zip(rs, rl):
                    torch.autograd.grad(iic_b200.sup_kl_from_logits(a_, l_, return_dice=True)[0], (a_,))

            def uda_rot():
                for a_, t_ in zip(rs, rt):
                    torch.autograd.grad(iic_b200.uda_from_logits(a_, t_, "mse"), (a_,))

            def flip_uda_rot():
                for a_, t_ in zip(rs, rt):
                    torch.autograd.grad(iic_b200.uda_from_logits(a_, t_, "mse", teacher_flips=rf), (a_,))

            def flip_rot():
                for t_ in rt:
                    iic_b200.flip_stack(t_, rf)

            def ref_flip_seq():
                tf = torch.stack([x_.clone().flip([d for d, bit in ((1, 1), (2, 2)) if f & bit]) if f else x_.clone()
                                  for x_, f in zip(rt[0], fl)], dim=0)
                return torch.autograd.grad(iic_b200.uda_from_logits(rs[0], tf, "mse"), (rs[0],))

            px_ = B * H * W
            ms_a, ms_u, ms_b, ms_c = (timed_graph(f_) / NR for f_ in (sup_rot, uda_rot, flip_uda_rot, flip_rot))
            extra["section_8f_kernels_from_hbm"] = {
                "what": "supervised KL + Dice (12*C+16 B/px), UDA mse from logits (20*C B/px), UDA through flips (20*C B/px) and "
                        "flip_stack (8*C B/px) at (B,4,H,W), fwd+bwd, inputs rotating over 4 sets inside one graph replay so "
                        "they come from HBM; fractions of the measured HBM copy bandwidth",
                "supervised_ms": round(ms_a, 4), "supervised_hbm_frac": round(64.0 * px_ / (ms_a * 1e-3) / 1e9 / hbm_peak, 4),
                "uda_ms": round(ms_u, 4), "uda_hbm_frac": round(80.0 * px_ / (ms_u * 1e-3) / 1e9 / hbm_peak, 4),
                "uda_flip_ms": round(ms_b, 4), "uda_flip_hbm_frac": round(80.0 * px_ / (ms_b * 1e-3) / 1e9 / hbm_peak, 4),
                "flip_stack_ms": round(ms_c, 4), "flip_stack_hbm_frac": round(32.0 * px_ / (ms_c * 1e-3) / 1e9 / hbm_peak, 4),
                "torch_flip_stack_plus_uda_ms": round(timed_graph(ref_flip_seq), 4)}
            del rs, rt, rl
        except Exception as e:  # noqa: BLE001
            extra["section_8f_from_hbm_error"] = f"{type(e).__name__}: {e}"
        if world == 1:
            try:
                # the other BASELINE configurations, per-GPU shapes, whole workload steps (device-timed graph replays)
                for cid in (3, 4, 5):
                    wl_ = WORKLOADS[cid]
                    B_ = batch_of(wl_, 8)
                    with contextlib.redirect_stdout(sys.stderr):
                        cr_ = [iic_b200.IIDSegmentationSmallPathLoss(padding=p_, patch_size=ps_) if k_ == "local" else iic_b200.IIDLoss()
                               for k_, S_, K_, H_, W_, p_, ps_, w_ in wl_["groups"]]
                    st_ = build_step(wl_, B_, cr_, iic_b200.iic_losses, uda_fn, torch)
                    ts_ = [t_.requires_grad_(m) for t_, m in zip(make_inputs(torch, dev, 4000 + cid, wl_, B_), grad_mask(wl_))]
                    ms_ = timed_graph(lambda: st_(ts_), reps=5)
                    px__ = pixels_per_step(wl_, B_)
                    algb = 24.0 * sum(S_ * K_ * B_ * (H_ * W_ if k_ == "local" else 1) for k_, S_, K_, H_, W_, p_, ps_, w_ in wl_["groups"])
                    flops = sum(6.0 * K_ * K_ * (2 * p_ + 1) ** 2 * S_ * B_ * H_ * W_ for k_, S_, K_, H_, W_, p_, ps_, w_ in wl_["groups"] if k_ == "local")
                    extra[f"config{cid}_per_gpu_step"] = {
                        "what": wl_["name"] + f" -- the per-GPU share at 8 GPUs (B = {B_}), one workload step in a CUDA graph, ONE finish "
                                              "launch for all terms; run `bench.py --config %d --gpus N` for the scaling line" % cid,
                        "ms": round(ms_, 4), "mpx_s": round(px__ / (ms_ * 1e-3) / 1e6, 1),
                        "hbm_frac": round(algb / (ms_ * 1e-3) / 1e9 / hbm_peak, 4),
                        "fp32_equiv_tflops": round(flops / (ms_ * 1e-3) / 1e12, 1),
                        "tensor_frac_of_measured_tf32_equiv_peak": round(2 * flops / (ms_ * 1e-3) / 1e12 / (bf16_peak / 2.0), 4)}
                    del ts_, st_
                    torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001
                extra["configs_345_error"] = f"{type(e).__name__}: {e}"
            try:
                if os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "reference", "semi_seg")):
                    extra["udaiic_iteration"] = udaiic_iteration_extra(dev)
                    iic_b200.set_check_mode("deferred")
                else:
                    extra["udaiic_iteration"] = {"skipped": "oracle/_ref/reference absent (run oracle/make_ref.py where /root/reference exists)"}
            except Exception as e:  # noqa: BLE001
                extra["udaiic_iteration"] = {"error": f"{type(e).__name__}: {e}"}
                iic_b200.set_check_mode("deferred")

    # ---- end to end through the public API with HOST buffers (pinned, first-touched on the GPU's NUMA node) ----
    host = [t_.detach().cpu().pin_memory() for t_ in sets[0]]
    # a training loop prefetches the next batch while the current one is computed: two device staging sets, the H2D copies
    # on their own stream, the D2H of the gradients on a third (PCIe is full duplex); every step still moves all of its
    # inputs from pinned host memory and reads its result back, inside the timed region
    stages = [[torch.empty_like(h, device=dev) for h in host] for _ in range(2)]
    gmask = grad_mask(wl)
    hloss = torch.empty((), dtype=torch.float32).pin_memory()
    hgrads = [torch.empty_like(h).pin_memory() for h, m in zip(host, gmask) if m]
    h2d = sum(h.numel() * 4 for h in host)
    d2h_grads = sum(h.numel() * 4 for h in hgrads)
    copy_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    e2e_i = [0]

    def e2e_step(with_grads):
        cur = torch.cuda.current_stream(dev)
        b = e2e_i[0] & 1
        e2e_i[0] += 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])            # the step before last has finished with this staging set
            for d_, h_ in zip(stages[b], host):
                d_.copy_(h_, non_blocking=True)
            ready[b].record(copy_stream)
        cur.wait_event(ready[b])
        ins = [d_.detach().requires_grad_(m) for d_, m in zip(stages[b], gmask)]
        loss, grads = step_fn(ins)
        consumed[b].record(cur)
        hloss.copy_(loss.detach(), non_blocking=True)
        if with_grads:
            d2h_stream.wait_stream(cur)
            with torch.cuda.stream(d2h_stream):
                for hg, g_ in zip(hgrads, grads):
                    g_.record_stream(d2h_stream)
                    hg.copy_(g_, non_blocking=True)

    def time_e2e(with_grads, n):
        for _ in range(3):
            e2e_step(with_grads)
        barrier()
        f0, f1 = ev(), ev()
        f0.record()
        for _ in range(n):
            e2e_step(with_grads)
        torch.cuda.current_stream(dev).wait_stream(d2h_stream)      # the last step's gradient copies end inside the timed region
        torch.cuda.current_stream(dev).wait_stream(copy_stream)
        f1.record()
        barrier()
        te = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return float(te.item()) / n

    e2e_steps = min(args.steps, 20)
    e2e_ms = time_e2e(False, e2e_steps)
    e2e_ms_g = time_e2e(True, e2e_steps)
    iic_b200.raise_if_flagged(dev)

    # ---- nothing after the measurements may be able to hang the job (graphs with captured exchange kernels alive):
    # multi-rank runs end with a barrier, the JSON line and a hard exit ----
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()
    watchdog = threading.Timer(400.0, lambda: os._exit(0))
    watchdog.daemon = True
    watchdog.start()

    if rank == 0:
        try:
            cpu = cpu_reference_run(args.config, world, 3, 1, budget_s=25.0)
            cpu_line = {"value": round(cpu["value"], 4), "unit": UNIT, "cores": cpu["threads"], "kind": cpu["kind"],
                        "sample": cpu["sample"], "best_ms": round(cpu["best_ms"], 2)}
        except Exception as e:  # noqa: BLE001
            cpu_line = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "unavailable", "sample": f"{type(e).__name__}: {e}"}
        cfg = workload_config(args.config, world)
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4), "higher_is_better": True,
            "scaling": wl["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "timing": {"launch": "cuda_graph_replay" if use_graph else "eager",
                       "input_set_bytes": set_bytes, "input_sets": NSETS,
                       "checks": "deferred (device-side simplex + NaN flags, read after the timed region)",
                       "api": "iic_b200.iic_losses(every (criterion, x, y) of the step) + torch.autograd.grad",
                       "multi_gpu": ("batch sharded; ONE exchange of all fp64 joints per step inside the finish launch, transport = "
                                     + iic_b200.data_parallel_transport()) if world > 1 else "single GPU"},
            "e2e": {"value": round(px_job / (e2e_ms * 1e-3) / 1e6, 2), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(e2e_ms, 4), "steps": e2e_steps,
                    "d2h_note": "the loss only (what a training loop reads back); with_gradients also copies every input "
                                "gradient to the host",
                    "with_gradients": {"value": round(px_job / (e2e_ms_g * 1e-3) / 1e6, 2), "unit": UNIT,
                                       "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 + d2h_grads,
                                       "ms_per_step": round(e2e_ms_g, 4)},
                    "host_buffers": "pinned, allocated after binding the process to the GPU's NUMA node", "numa": numa,
                    "pipeline": "double-buffered: the H2D of step i+1 (own stream) overlaps the compute of step i; gradient D2H on a "
                                "third stream"},
            "gpu_launches": (n_own or static_launch_count(wl, world)) * args.steps,
            "gpu_launches_per_step": n_own or static_launch_count(wl, world),
            "gpu_launches_source": "counted with torch.profiler on one eager step" if n_own else "dispatch rules (profiler unavailable)",
            "gpu_kernels": own_names,
            "clocks": clocks,
            "roofline": roofline,
            "cpu_baseline": cpu_line,
            "multi_gpu_check": mg,
            "wall_s_timed_region": round(t_wall, 4),
            "extra": extra,
        }
        if dumped is not None:
            line["dumped_outputs"] = {"dir": os.path.abspath(args.dump_outputs), "step": args.steps - 1,
                                      "input_set": (args.steps - 1) % NSETS, "arrays": dumped}
        print(json.dumps(line), flush=True)
    watchdog.cancel()
    if world > 1:
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
