"""CPU check: the stand-alone kernel harnesses under tools/ still compile and link against the library's sources.

Each harness #includes one kernel family's .cu file and calls its entry point directly, so a signature change in
csrc/ that is not carried into the harnesses breaks them; this test catches that on a machine without a GPU.
The csrc harnesses link csrc/runtime.cu (error text, device queries, options); the experiment under
tools/experiments/ carries its own copies of those and builds alone."""
import importlib.util
import os
import subprocess

import pytest

from conftest import ROOT

PKG = os.path.join(ROOT, "mi-based-regularized-semi-supervised-segmentation_b200")
RUNTIME = os.path.join(PKG, "csrc", "runtime.cu")

# (harness, -D flags of its build line, links csrc/runtime.cu)
HARNESSES = [
    ("tools/tc_joint_harness.cu", [], True),
    ("tools/tc_jointp_harness.cu", [], True),
    ("tools/tc_joint10_harness.cu", ["-DIIC_TCJ_DEBUG"], True),
    ("tools/tc_bwd_harness.cu", [], True),
    ("tools/tc_bwdrb_harness.cu", [], True),
    ("tools/tc_bwdrb10_harness.cu", [], True),
    ("tools/tc_bwdrb10h_harness.cu", [], True),
    ("tools/tma_debug.cu", ["-DIIC_TMA_DEBUG"], True),
    ("tools/experiments/tc_jointp10_harness.cu", [], False),
]


def _build_module():
    spec = importlib.util.spec_from_file_location("iic_b200_build", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("harness,defines,with_runtime", HARNESSES, ids=[os.path.basename(h[0]) for h in HARNESSES])
def test_harness_builds(harness, defines, with_runtime, tmp_path):
    build = _build_module()
    try:
        nvcc = build._nvcc()
    except RuntimeError:
        pytest.skip("nvcc not found")
    srcs = [os.path.join(ROOT, harness)] + ([RUNTIME] if with_runtime else [])
    exe = str(tmp_path / "harness")
    r = subprocess.run([nvcc, *build.NVCC_FLAGS, *defines, "-o", exe, *srcs], capture_output=True, text=True,
                       cwd=tmp_path)
    assert r.returncode == 0, f"{harness} does not build:\n{r.stdout}\n{r.stderr}"
    assert os.path.exists(exe)
