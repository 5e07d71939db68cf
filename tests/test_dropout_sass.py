"""CPU test (no GPU): adding the dropout forms of the classifier kernels and moving the Philox block into common.cuh leave
the machine code of the existing classifier GEMMs (k_gemm<*,*>, k_gemm_s<*,*>), classifier loss kernels and the fused
selection kernel unchanged.  tests/golden/dropout_sass.json holds the sha256 of their SASS (instructions and encodings,
addresses stripped) as the recorded nvcc release compiles them with the library's flags; another nvcc release may
schedule differently, so the test skips there.  The digests of k_loss_rows and k_loss_rows2 were re-recorded once, when
their cross-entropy terms changed to keep log-sum-exp relative to the row maximum (csrc/loss_optim.cu CE_LSE_NOTE);
every other function keeps the digest recorded before the dropout forms were added."""
import json
import os
import subprocess

import pytest

from test_step_tail_sass import _tool, sass_digests

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "dropout_sass.json")
NEW_KERNELS = {
    "gcn.cu": ["k_gemm_dropout<true>", "k_gemm_dropout<false>", "k_gemm_s_dropout<true>", "k_gemm_s_dropout<false>"],
    "loss_optim.cu": ["k_loss_rows2_dropout", "k_loss_final2_dropout", "k_loss_rows_dropout", "k_loss_final_dropout",
                      "k_dropout_mask"],
    "select.cu": [],
}


def _demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return {n: d.split("(")[0].replace("void ", "") for n, d in zip(names, out)}


def test_classifier_and_selection_kernels_keep_their_recorded_sass(tmp_path):
    nvcc, cuobjdump = _tool("nvcc"), _tool("cuobjdump")
    if not nvcc or not cuobjdump:
        pytest.skip("nvcc / cuobjdump not available")
    golden = json.load(open(GOLDEN))
    ver = subprocess.run([nvcc, "--version"], capture_output=True, text=True).stdout
    if golden["nvcc"] not in ver:
        pytest.skip(f"SASS recorded with nvcc {golden['nvcc']}")
    from grapes_b200.build import NVCC_FLAGS
    for src, new in NEW_KERNELS.items():
        cubin = str(tmp_path / (src + ".cubin"))
        subprocess.run([nvcc] + NVCC_FLAGS + ["-cubin", "-o", cubin, os.path.join(ROOT, "grapes_b200", "csrc", src)],
                       check=True, capture_output=True)
        got = sass_digests(subprocess.run([cuobjdump, "-sass", cubin], check=True, capture_output=True, text=True).stdout)
        for name, rec in golden["functions"].items():
            if rec["file"] == src:
                assert got.get(name) == rec["sha256"], f"SASS of {name} changed"
        if new:
            present = set(_demangle(sorted(got)).values())
            for k in new:
                assert k in present, f"{k} missing from {src}"
