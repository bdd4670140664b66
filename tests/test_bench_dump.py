"""bench.py --dump-outputs: what it writes for a step's outputs, on the CPU."""
import os

import numpy as np
import torch

import bench


def test_output_names_cover_every_step_output():
    for wl in bench.WORKLOADS.values():
        names = bench.output_names(wl)
        assert len(names) == len(set(names)) == 1 + sum(bench.grad_mask(wl))


def test_dump_outputs_sampled_reproducible_and_bounded(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 5000)              # 5000 float32 values in all
    wl = bench.WORKLOADS[2]
    g = torch.Generator().manual_seed(0)
    grads = [torch.randn(s, generator=g) for s in ((2, 10, 30, 40), (2, 10, 30, 40), (32, 10), (32, 10))]
    loss = torch.tensor(0.25)
    a = bench.dump_outputs(str(tmp_path / "a"), wl, loss, grads)
    b = bench.dump_outputs(str(tmp_path / "b"), wl, loss, grads.copy())
    assert a == b and list(a) == bench.output_names(wl)
    assert a["grad_1_global_y"] == {"numel": 320, "written": 320}
    # what the small arrays leave unused goes to the large ones
    assert [a[n]["written"] for n in ("grad_0_local_x", "grad_0_local_y")] == [2179, 2180]
    total = 0
    for name in bench.output_names(wl):
        x, y = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert x.dtype == np.float32 and np.array_equal(x, y)
        total += x.nbytes
    assert total == bench.DUMP_BYTES
    assert np.load(tmp_path / "a" / "loss.npy").tolist() == [0.25]
    assert np.array_equal(np.load(tmp_path / "a" / "grad_1_global_x.npy"), grads[2].numpy().reshape(-1))
    sample = np.load(tmp_path / "a" / "grad_0_local_x.npy")
    assert np.isin(sample, grads[0].numpy()).all() and len(np.unique(sample)) == 2179
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in bench.output_names(wl))
