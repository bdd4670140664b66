"""CPU-side checks: the C-ABI library loads and exports every declared symbol, the host mirror keeps the
reference's API surface, and nothing silently falls back to the CPU."""
import inspect
import os
import re
import sys

import pytest
import torch

from conftest import ROOT, load_golden

PKG = os.path.join(ROOT, "mi-based-regularized-semi-supervised-segmentation_b200")
REF_MISSING = "the original project's source is not provided (IIC_REFERENCE_ROOT or oracle/_ref/reference)"


@pytest.fixture(scope="module")
def built():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as ge
    ge.build()
    import iic_b200
    return iic_b200


def test_library_exports_every_declared_symbol(built):
    import ctypes
    hdr = open(os.path.join(ROOT, "include", "iic_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(iic_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 15
    lib = ctypes.CDLL(os.path.join(PKG, "libiic_b200.so"))
    for name in declared:
        assert hasattr(lib, name), f"libiic_b200.so does not export {name}"
    assert declared == set(built._lib.PROTOTYPES), declared ^ set(built._lib.PROTOTYPES)
    declared_abi = int(re.search(r"#define IIC_B200_ABI_VERSION (\d+)", hdr).group(1))
    assert built._lib.load().iic_b200_abi_version() == built._lib.ABI_VERSION == declared_abi


def test_options_are_read_once_and_settable(built):
    """The dispatch switches are a table inside the library (csrc/runtime.cu): environment defaults are read once,
    iic_b200_set_option changes them afterwards, unknown names are errors."""
    L = built._lib
    lib = L.load()
    assert lib.iic_b200_get_option(b"tcrb_p1") in (0, 1)
    old = L.set_option("tcrb_p1", 1)
    try:
        assert lib.iic_b200_get_option(b"tcrb_p1") == 1
        os.environ["IIC_B200_TCRB_P1"] = "0"          # too late: the environment was read at first use
        assert lib.iic_b200_get_option(b"tcrb_p1") == 1
    finally:
        os.environ.pop("IIC_B200_TCRB_P1", None)
        L.set_option("tcrb_p1", old)
    assert lib.iic_b200_get_option(b"xchg_timeout_ms") > 0
    # every documented switch (INTEGRATION.md) exists in the table
    for name in ("no_tma", "no_tc", "no_tc10", "no_tcj10", "no_fast", "tcp_p1", "tcrb_p1", "tc10_force", "tc10_tf32",
                 "no_fused_epilogue", "fin_last_cta_epilogue", "xchg_timeout_ms"):
        assert lib.iic_b200_get_option(name.encode()) >= 0, name
    assert lib.iic_b200_set_option(b"no_such_switch", 1) != 0
    assert lib.iic_b200_get_option(b"no_such_switch") == -1
    # the coefficient buffers carry the tensor-core weight images: no hidden allocation in the backward
    assert lib.iic_local_coeff_floats(10, 1, 1) == 10 * 9 * 12
    assert lib.iic_local_coeff_floats(20, 3, 1) > 20 * 49 * 20
    assert lib.iic_local_coeff_floats(128, 1, 1) > 128 * 9 * 128
    assert lib.iic_local_coeff_floats(20, 3, 4) == 4 * 20 * 49 * 20       # several patches: generic kernels only


def test_patch_count_matches_reference_windows(built):
    lib = built._lib.load()
    g = load_golden("patch_windows")
    for key, wins in g.items():
        hw, ps = key.split("_p")
        h, w = (int(v) for v in hw.split("x"))
        ps = int(ps)
        assert lib.iic_local_num_patches(h, w, ps, ps, ps // 2, ps // 2) == len(wins), key
    assert lib.iic_local_num_patches(10, 10, 4, 4, 0, 0) == -1      # step 0 with patch < map is an error


def test_api_surface_matches_reference(built):
    iic = built
    sig = inspect.signature
    assert list(sig(iic.IIDLoss.__init__).parameters) == ["self", "lamb", "eps"]
    assert list(sig(iic.IIDLoss.forward).parameters) == ["self", "x_out", "x_tf_out"]
    assert list(sig(iic.compute_joint).parameters) == ["x_out", "x_tf_out", "symmetric"]
    assert list(sig(iic.IIDSegmentationLoss.__init__).parameters) == ["self", "lamda", "padding", "eps"]
    assert sig(iic.IIDSegmentationLoss.__init__).parameters["padding"].default == 7
    assert list(sig(iic.IIDSegmentationLoss.__call__).parameters) == ["self", "x_out", "x_tf_out", "mask"]
    assert list(sig(iic.IIDSegmentationSmallPathLoss.__init__).parameters) == ["self", "lamda", "padding", "eps",
                                                                               "patch_size"]
    assert sig(iic.IIDSegmentationSmallPathLoss.__init__).parameters["patch_size"].default == 32
    assert list(sig(iic.patch_generator).parameters) == ["feature_map", "patch_size", "step_size"]
    assert list(sig(iic.KL_div.__init__).parameters) == ["self", "reduction", "eps", "weight", "verbose"]
    m = iic.IIDLoss(lamb=2.0)
    assert m.lamb == 2.0 and hasattr(m, "eps") and m.torch_vision == torch.__version__
    w = iic.IICLossWrapper(["Conv5", "Up_conv3", "Up_conv2"], [1, 3], [1024, 1024])
    assert w.feature_names == ["Conv5", "Up_conv3", "Up_conv2"]
    assert type(w["Conv5"]).__name__ == "IIDLoss" and w["Up_conv2"].padding == 3
    assert [k for k, _ in w.items()] == ["Conv5", "Up_conv3", "Up_conv2"]
    with pytest.raises(IndexError):
        w["Conv1"]


def test_patch_generator_views(built):
    g = load_golden("patch_windows")
    for key, wins in g.items():
        hw, ps = key.split("_p")
        h, w = (int(v) for v in hw.split("x"))
        ps = int(ps)
        fm = torch.arange(h * w, dtype=torch.float32).reshape(1, 1, h, w)
        got = [(int(p[0, 0, 0, 0]) // w, int(p[0, 0, 0, 0]) // w + p.shape[2], int(p[0, 0, 0, 0]) % w,
                int(p[0, 0, 0, 0]) % w + p.shape[3]) for p in built.patch_generator(fm, (ps, ps), (ps // 2, ps // 2))]
        assert got == [tuple(r) for r in wins.tolist()]


def test_no_cpu_fallback(built):
    x = torch.rand(2, 4, 8, 8).softmax(1).requires_grad_(True)
    with pytest.raises(Exception) as ei:
        built.IIDSegmentationLoss(padding=1)(x, x.detach().clone().requires_grad_(True))
    assert "CPU" in str(ei.value) or "CUDA" in str(ei.value)
    with pytest.raises(Exception):
        built.MSELoss()(x, x.detach())
    with pytest.raises(Exception) as ei:
        built.sup_kl_from_logits(torch.randn(2, 4, 8, 8, requires_grad=True), torch.zeros(2, 8, 8, dtype=torch.int64))
    assert "CPU" in str(ei.value) or "CUDA" in str(ei.value)


def test_flip_flags_replay_the_reference_draws(built):
    """draw_flip_flags == the draws of the reference's seeded per-sample loop (golden fixtures made by running it)."""
    from conftest import golden_names
    names = golden_names("flip")
    assert names
    for name in names:
        g = load_golden(name)
        flags = built.draw_flip_flags(int(g["seed"]), len(g["teacher"]))
        assert flags.dtype == torch.uint8 and flags.tolist() == g["flags"].tolist(), name
    assert built.draw_flip_flags(5, 4, axis=None).tolist() == [0, 0, 0, 0]
    assert built.TensorRandomFlip(axis=[1, 2], threshold=0.8).flags(3, 8).tolist() == load_golden("f_8x4x6x8_mse")["flags"].tolist()
    with pytest.raises(ValueError):
        built.draw_flip_flags(0, 2, axis=[0])
    import random
    state = random.getstate()
    built.draw_flip_flags(123, 16)
    assert random.getstate() == state          # like FixRandomSeed, the module-level generator is left alone
    with pytest.raises(Exception) as ei:       # no CPU path for the kernels themselves
        built.flip_stack(torch.zeros(2, 1, 4, 4), 0)
    assert "CPU" in str(ei.value) or "CUDA" in str(ei.value)


def test_flip_flags_against_live_reference(built):
    """Many seeds, batch sizes, axes and thresholds against the reference's own TensorRandomFlip loop.  Needs the original
    project's source: no reference draws are stored for a non-default axis or threshold."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_loader
    if not ref_loader.available():
        pytest.skip(REF_MISSING)
    TensorRandomFlip, FixRandomSeed = ref_loader.load_flip()
    for axis, thr in (([1, 2], 0.8), ([2], 0.5), ([1], 0.3), ([2, 1], 0.8)):
        T = TensorRandomFlip(axis=axis, threshold=thr)
        for seed in (0, 1, 2, 17, 4242, 2**31 - 1):
            for B in (1, 5, 10):
                x = torch.arange(B * 2 * 3 * 4, dtype=torch.float32).reshape(B, 2, 3, 4)
                with FixRandomSeed(seed):
                    ref = torch.stack([T(s) for s in x], dim=0)
                flags = built.draw_flip_flags(seed, B, axis, thr).tolist()
                mine = torch.stack([s.flip([d for d, bit in ((1, 1), (2, 2)) if f & bit]) if f else s
                                    for s, f in zip(x, flags)], dim=0)
                assert torch.equal(mine, ref), (axis, thr, seed, B)


def test_sub_head_and_layer_reductions(built):
    """A7 of SURVEY.md section 8a: the epocher's two reductions and their batched form."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import iic_oracle as O
    from iic_b200.semi_seg._utils import average_iter, combine_iic_losses, weighted_average_iter
    torch.manual_seed(0)
    layers = [[torch.randn((), dtype=torch.float64, requires_grad=True) for _ in range(n)] for n in (5, 5, 3)]
    imp = [0.5, 0.3, 0.2]
    means = [average_iter(h) for h in layers]
    ref = weighted_average_iter(means, imp)
    want = O.weighted_average_iter([O.average_iter([float(l.detach()) for l in h]) for h in layers], imp)
    assert abs(ref.item() - want) < 1e-14
    total, per_layer = combine_iic_losses(layers, imp)
    assert abs(total.item() - want) < 1e-14
    assert torch.allclose(per_layer, torch.stack([m.detach() for m in means]), atol=1e-15)
    total.backward()                                   # d total / d loss = importance / (sum + 1e-16) / heads
    assert abs(float(layers[2][1].grad) - 0.2 / (1.0 + 1e-16) / 3) < 1e-15


def test_batched_cluster_heads_match_reference(built):
    """iic_b200.trainer heads load the reference heads' state_dict (strict) and give the same maps and gradients
    (contrastyou/trainer/_utils.py:96-168, loaded by path from the original project's source when it is provided; no
    outputs of the reference heads are stored, so without it this comparison is not made)."""
    import importlib.util
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_loader
    path = os.path.join(ref_loader.REFERENCE_ROOT, "contrastyou", "trainer", "_utils.py")
    if not os.path.isfile(path):
        pytest.skip(REF_MISSING)
    spec = importlib.util.spec_from_file_location("_ref_trainer_utils", path)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    from iic_b200.trainer import ClusterHead, LocalClusterHead
    torch.manual_seed(0)
    for kw in (dict(head_type="linear", num_clusters=10, num_subheads=5, T=1, normalize=False),
               dict(head_type="linear", num_clusters=7, num_subheads=3, T=0.5, normalize=True),
               dict(head_type="mlp", num_clusters=6, num_subheads=2, T=1, normalize=False)):
        for ref_cls, cls, shape in ((ref.LocalClusterHead, LocalClusterHead, (4, 16, 12, 10)),
                                    (ref.ClusterHead, ClusterHead, (6, 16, 5, 5))):
            r, m = ref_cls(16, **kw).double(), cls(16, **kw).double()
            m.load_state_dict(r.state_dict(), strict=True)
            f1 = torch.randn(*shape, dtype=torch.float64, requires_grad=True)
            f2 = f1.detach().clone().requires_grad_(True)
            o1, o2 = r(f1), m(f2)
            assert len(o1) == len(o2) == kw["num_subheads"]
            assert max((a - b).abs().max().item() for a, b in zip(o1, o2)) < 1e-14
            w = [torch.randn_like(o) for o in o1]
            sum((a * c).sum() for a, c in zip(o1, w)).backward()
            sum((a * c).sum() for a, c in zip(o2, w)).backward()
            assert (f1.grad - f2.grad).abs().max().item() < 1e-13
            assert max((p.grad - q.grad).abs().max().item() for p, q in zip(r.parameters(), m.parameters())) < 1e-12
            lg = m.logits(f2.detach())
            assert all(torch.allclose(torch.softmax((torch.nn.functional.normalize(z, p=2, dim=1) if kw["normalize"]
                                                     else z) / kw["T"], 1), o.detach(), atol=1e-14)
                       for z, o in zip(lg, o2)) or kw["normalize"]
            assert all(o.stride(-1) == 1 for o in o2)          # what the loss kernels require of their inputs


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(PKG):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("the oracle", ""), f"{f} mentions the oracle"


def test_deferred_scalar_meters_match_average_value_meter(built):
    """DeferredScalarMeters (SURVEY 8f row 3): same means as dc2's AverageValueMeter fed with .item() values, NaN for a
    name that was never recorded, buffer roll-over, reset."""
    torch.manual_seed(0)
    m = built.DeferredScalarMeters(["sup_loss", "reg_loss", "uda", "never"], capacity=4)
    vals = torch.randn(11, 3)
    for r in vals:
        m.record(sup_loss=r[0], reg_loss=r[1], uda=float(r[2]))       # tensors and plain numbers
    s = m.summary()
    for i, n in enumerate(["sup_loss", "reg_loss", "uda"]):
        assert abs(s[n]["mean"] - vals[:, i].double().mean().item()) < 1e-6
    assert s["never"]["mean"] != s["never"]["mean"]                     # NaN
    m.reset()
    m.record(sup_loss=torch.tensor(2.0))
    assert m.summary()["sup_loss"]["mean"] == 2.0
    with pytest.raises(AssertionError):
        m.record(bogus=1.0)
