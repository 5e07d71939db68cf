"""CPU test (no GPU): adding the int64 row-slab form of the whole-graph aggregation (template parameter W64 of k_agg and
k_agg_tma, grapes_aggregate_rows64) leaves the machine code of every existing aggregation kernel unchanged.
tests/golden/agg_sass.json holds the sha256 of their SASS (instructions and encodings, addresses stripped) as the recorded
nvcc release compiled them before W64 existed, keyed by demangled name; the same kernel now carries `, false` as its last
template argument.  Another nvcc release may schedule differently, so the test skips there."""
import json
import os
import subprocess

import pytest

from test_dropout_sass import _demangle
from test_step_tail_sass import _tool, sass_digests

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "agg_sass.json")
NEW_KERNELS = {
    "gcn.cu": [f"k_agg<{v}, {b}, true>" for v in (1, 2, 4) for b in ("false", "true")],
    "spmm_tma.cu": ["k_agg_tma<1, false, 1, false, true>", "k_agg_tma<2, false, 1, false, true>",
                    "k_agg_tma<5, false, 1, false, true>", "k_agg_tma<12, false, 1, false, true>",
                    "k_agg_tma<1, false, 1, true, true>", "k_agg_tma<2, false, 1, true, true>"],
}


def _current_name(recorded: str) -> str:
    return recorded if recorded.startswith("k_agg_rows<") else recorded[:-1] + ", false>"


def test_existing_aggregation_kernels_keep_their_sass(tmp_path):
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
        by_name = {d: got[m] for m, d in _demangle(sorted(got)).items()}
        recorded = {k: r for k, r in golden["functions"].items() if r["file"] == src}
        assert recorded
        for name, rec in recorded.items():
            assert by_name.get(_current_name(name)) == rec["sha256"], f"SASS of {name} changed"
        for k in new:
            assert k in by_name, f"{k} missing from {src}"
